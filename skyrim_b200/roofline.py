"""Algorithmic work of one 6-h step, per kernel family (the figures bench.py's ``roofline``
object and DESIGN.md use; derivation in SURVEY.md §8(d)).  FLOPs are 2*MAC of the dense
contractions; bytes are the mandatory HBM traffic of the family's fused kernel."""
from __future__ import annotations

from .config import FCNConfig, PanguConfig, SFNOConfig

WIN_TOK = 144


def pangu_flops(cfg: PanguConfig) -> dict:
    C = cfg.dim
    HW = cfg.H * cfg.W
    T1, T2 = cfg.Z * HW, cfg.Z * cfg.H2 * cfg.W2
    nwin1 = (cfg.Z // 2) * (cfg.padded_h(cfg.H) // 6) * (cfg.W // 12)
    nwin2 = (cfg.Z // 2) * (cfg.padded_h(cfg.H2) // 6) * (cfg.W2 // 12)
    f = dict(qkv=0.0, attn=0.0, proj=0.0, fc1=0.0, fc2=0.0)
    for li, depth in enumerate(cfg.depths):
        c, T, rows = (C, T1, nwin1 * WIN_TOK) if li in (0, 3) else (2 * C, T2, nwin2 * WIN_TOK)
        f["qkv"] += depth * 2.0 * rows * c * 3 * c
        f["attn"] += depth * 2.0 * 2.0 * rows * WIN_TOK * c
        f["proj"] += depth * 2.0 * rows * c * c
        f["fc1"] += depth * 2.0 * T * c * 4 * c
        f["fc2"] += depth * 2.0 * T * 4 * c * c
    f["mlp"] = f["fc1"] + f["fc2"]
    nzt = cfg.Z - 1
    f["embed"] = 2.0 * nzt * HW * 160 * C + 2.0 * HW * 112 * C
    f["recover"] = 2.0 * nzt * HW * 2 * C * 160 + 2.0 * HW * 2 * C * 64
    f["down"] = 2.0 * T2 * 4 * C * 2 * C
    f["up"] = 2.0 * T2 * 2 * C * 4 * C + 2.0 * T1 * C * C
    f["total"] = (f["qkv"] + f["attn"] + f["proj"] + f["fc1"] + f["fc2"] + f["embed"] + f["recover"]
                  + f["down"] + f["up"])
    return f


def pangu_bytes(cfg: PanguConfig) -> dict:
    """Mandatory HBM bytes per 6-h step and kernel family for the DEFAULT data flow of DESIGN.md section 3 (the token stream
    exists only as its fp16 operand image xh; weights stay in L2 and are not counted).  Per token and feature:
      qkv    read xh 2 B, write q|k|v window images 3 x 2 B (padded tokens included)
      attn   read q|k|v 6 B, write the projection's operand image 2 B
      proj   read operand image 2 B, residual read from xh 2 B, xh written in place 2 B
      mlp    read xh 2 B (operand; the epilogue re-reads the same image as the residual: an L2 hit, ncu profiles/r2f_traffic.json),
             xh written in place 2 B (the 4C hidden activation never leaves the SM)
    (with the fp32 token stream, "fp32_stream", proj and mlp move 12 B)"""
    C = cfg.dim
    HW = cfg.H * cfg.W
    T1, T2 = cfg.Z * HW, cfg.Z * cfg.H2 * cfg.W2
    nwin1 = (cfg.Z // 2) * (cfg.padded_h(cfg.H) // 6) * (cfg.W // 12)
    nwin2 = (cfg.Z // 2) * (cfg.padded_h(cfg.H2) // 6) * (cfg.W2 // 12)
    b = dict(qkv=0.0, attn=0.0, proj=0.0, mlp=0.0)
    for li, depth in enumerate(cfg.depths):
        c, T, rows = (C, T1, nwin1 * WIN_TOK) if li in (0, 3) else (2 * C, T2, nwin2 * WIN_TOK)
        b["qkv"] += depth * (2.0 * T * c + 6.0 * rows * c)
        b["attn"] += depth * (6.0 * rows * c + 2.0 * T * c)
        b["proj"] += depth * 6.0 * T * c
        b["mlp"] += depth * 4.0 * T * c
    state = float(pangu_state_bytes(cfg))
    b["embed"] = state + T1 * C * (4.0 + 2.0)                  # state in; x (fp32) + operand image out
    b["recover"] = 2.0 * T1 * C * 2.0 + state                  # concat(skip, x) images in; state out
    b["down"] = T1 * C * 2.0 + T2 * 4 * C * 2.0 * 2 + T2 * 2 * C * 2.0           # image in, merged image out + in, image out
    b["up"] = T2 * 2 * C * 2.0 + T1 * C * 2.0 * 2 + T1 * C * 2.0                 # image in, shuffled image out + in, image out
    b["total"] = sum(b.values())
    return b


def pangu_state_bytes(cfg: PanguConfig) -> int:
    return cfg.n_channels * cfg.nlat * cfg.nlon * 4


def sfno_flops(cfg: SFNOConfig) -> dict:
    """SURVEY.md §8(d) formulae (Legendre contractions, per-l channel mixing, pixel MLPs); the
    longitude DFT is counted as an FFT (negligible) although the engine runs it as a GEMM, and
    the 3-term fp16 split triples the executed tensor work without changing these figures."""
    E, Cin, L = cfg.embed, cfg.n_channels, cfg.layers
    P1, P2 = cfg.nlat * cfg.nlon, cfg.h * cfg.w
    lm = cfg.lmax * cfg.mmax
    f = {}
    f["sfno_enc"] = 2.0 * P1 * (Cin * E + E * E)
    f["sfno_dec"] = 2.0 * P1 * ((E + Cin) * E + E * Cin)
    leg_big, leg_int = 4.0 * cfg.nlat * lm * E, 4.0 * cfg.h * lm * E
    f["sfno_sht"] = leg_big + (L - 1) * leg_int
    # inverse transforms: mixed spectrum of every block + the resampled residual of the two grid-changing blocks
    f["sfno_isht"] = (L - 1) * leg_int + leg_big + leg_int + leg_big
    f["sfno_spec"] = L * 8.0 * lm * E * E
    mlp_int = 2.0 * P2 * (E * E + 2 * cfg.mlp_ratio * E * E)
    mlp_big = 2.0 * P1 * (E * E + 2 * cfg.mlp_ratio * E * E)
    f["sfno_mlp"] = (L - 1) * mlp_int + mlp_big
    f["total"] = sum(f.values())
    return f


def sfno_bytes(cfg: SFNOConfig) -> dict:
    """Mandatory HBM bytes per step and family with fp32 activations between stages (E channels; pixels P1 at 721x1440,
    P2 on the internal grid); spectral weights are streamed once per step and layer."""
    E, Cin, L = cfg.embed, cfg.n_channels, cfg.layers
    P1, P2 = cfg.nlat * cfg.nlon, cfg.h * cfg.w
    lm = cfg.lmax * cfg.mmax
    b = {}
    b["sfno_enc"] = 4.0 * P1 * (Cin + E) + 4.0 * P1 * E          # state in, x out, positional embedding in
    b["sfno_dec"] = 4.0 * P1 * (E + Cin + Cin)
    b["sfno_sht"] = 4.0 * E * (P1 + (L - 1) * P2) + 8.0 * L * E * lm
    b["sfno_isht"] = 8.0 * (L + 2) * E * lm + 4.0 * E * (2 * P1 + L * P2)
    b["sfno_spec"] = L * (8.0 * cfg.lmax * E * E + 16.0 * E * lm)
    b["sfno_mlp"] = 4.0 * E * 4 * ((L - 1) * P2 + P1)
    b["total"] = sum(b.values())
    return b


def graphcast_counts(cfg, graph=None) -> dict:
    """row counts of the GraphCast step; without a graph, the full-size counts of the refinement-6 mesh"""
    if graph is not None:
        return dict(Ng=cfg.n_grid, Nm=int(graph["n_mesh"]), Em=len(graph["mesh.senders"]), Eg=len(graph["g2m.senders"]))
    assert (cfg.nlat, cfg.nlon, cfg.mesh_levels) == (721, 1440, 6)
    return dict(Ng=cfg.n_grid, Nm=40962, Em=327660, Eg=1629780)


def _graphcast_schedule(cfg, n):
    """The engine's per-step GEMM schedule (csrc/graphcast_engine.cu::step) as (family, rows, K, N, bytes per row):
    hidden GEMMs read their A operand image(s) (2 B per element) and write the 512-wide hidden image; LayerNorm GEMMs read
    the hidden image, read the residual (fp32 rows for mesh nodes, the stream's own fp16 image for grid nodes and mesh edges) and
    write the operand images listed."""
    L, F = cfg.latent, 192
    Ng, Nm, Em, Eg = n["Ng"], n["Nm"], n["Em"], n["Eg"]
    s = []
    # gathered per-node tables: a mesh-node table (<= 84 MB) stays in L2 and is counted once per GEMM; a grid-node table
    # (1 GB) is read from HBM per gathered row
    hid = lambda rows, K, grid_tab=0, mesh_tab=0: s.append(("gc_hidden", rows, K, L, 2.0 * K + 2.0 * L + grid_tab * 2.0 * L
                                                            + mesh_tab * Nm * 2.0 * L / rows))
    # residual: 0 none, 2 fp32 rows read + written (mesh nodes), 3 read from the stream's fp16 image (grid nodes, mesh edges)
    ln = lambda rows, res, img, yimg: s.append(("gc_ln", rows, L, L, 2.0 * L + (8.0 * L if res == 2 else 2.0 * L if res == 3 else 0.0)
                                                + 2.0 * L * (img + yimg)))
    tab = lambda rows, N: s.append(("gc_table", rows, L, N, 2.0 * L + 2.0 * N))
    hid(Ng, F); ln(Ng, 0, 1, 0)                                   # grid embedding
    tab(Ng, L); hid(Eg, L, grid_tab=1, mesh_tab=1); ln(Eg, 0, 0, 1)             # grid2mesh edges
    hid(Nm, 2 * L); ln(Nm, 2, 1, 0)                               # mesh nodes
    hid(Ng, L); ln(Ng, 3, 1, 0)                                   # grid nodes
    for i in range(cfg.layers):
        tab(Nm, 2 * L); hid(Em, L, mesh_tab=2)
        ln(Em, 3, 1, 1) if i < cfg.layers - 1 else ln(Em, 0, 0, 1)   # the last layer's edge latents are never read
        hid(Nm, 2 * L); ln(Nm, 2, 1, 0)
    tab(Nm, L); tab(Ng, L); hid(3 * Ng, L, grid_tab=1, mesh_tab=1); ln(3 * Ng, 0, 0, 1)   # mesh2grid edges
    hid(Ng, 4 * L); ln(Ng, 3, 1, 0)                               # grid update ([v | e0 | e1 | e2]: read as 4 images)
    hid(Ng, L)                                                    # output head, first layer
    return s


def graphcast_flops(cfg, graph=None) -> dict:
    """Dense FLOPs (2 MAC) of the step AS FORMULATED IN THE ENGINE — first layers split per input with per-node partial
    products (the published concatenated form needs ~26 TFLOP, this one ~18.5) — except that the mesh2grid grid update is
    counted with K = 2L (node + aggregated edges) although the engine contracts K = 4L (the three edge images separately)."""
    n = graphcast_counts(cfg, graph)
    f = dict(gc_hidden=0.0, gc_ln=0.0, gc_table=0.0, gc_feat=0.0, gc_agg=0.0)
    for fam, rows, K, N, _ in _graphcast_schedule(cfg, n):
        k_alg = 2 * cfg.latent if K == 4 * cfg.latent else (cfg.n_features if K == 192 else K)
        f[fam] += 2.0 * rows * k_alg * N
    f["gc_out"] = 2.0 * n["Ng"] * cfg.latent * cfg.n_state
    f["total"] = sum(f.values())
    return f


def graphcast_bytes(cfg, graph=None) -> dict:
    """Mandatory HBM bytes per step and kernel family for the engine's data flow (weights and the per-node tables are L2
    resident at mesh size and are counted once per GEMM)."""
    n = graphcast_counts(cfg, graph)
    L = cfg.latent
    b = dict(gc_hidden=0.0, gc_ln=0.0, gc_table=0.0)
    for fam, rows, K, N, per_row in _graphcast_schedule(cfg, n):
        b[fam] += rows * per_row
    plane = 4.0 * n["Ng"]
    b["gc_feat"] = plane * 2 * cfg.n_state + n["Ng"] * 192 * 2.0 + plane * (cfg.n_state + 1)    # state in; features, slice 0 and toa out
    b["gc_agg"] = (n["Eg"] + cfg.layers * n["Em"]) * 2.0 * L + (1 + cfg.layers) * n["Nm"] * 2.0 * L
    b["gc_out"] = n["Ng"] * 2.0 * L + plane * 2 * cfg.n_prog                                    # hidden in; x_t in, x_{t+1} out
    b["total"] = sum(b.values())
    return b


def fcn_flops(cfg: FCNConfig, batch: int = 1) -> dict:
    """FourCastNet v1 per step, by kernel family of csrc/fcn_engine.cu (fcn_ln does no contraction)"""
    M = batch * cfg.tokens
    E, K = cfg.embed, cfg.n_channels * cfg.patch ** 2
    lo, hi = cfg.h_range
    nk, kw, h, w = hi - lo, cfg.kw, cfg.h, cfg.w
    dft_w = 2 * (2.0 * batch * h * E * w * 2 * kw)                   # forward + inverse, real x complex
    dft_h = 2 * (8.0 * batch * kw * E * h * nk)                      # forward + inverse, complex
    block_mlp = 2 * (2.0 * batch * nk * kw * E * 2 * 2 * cfg.block_size)
    f = dict(fcn_embed=2.0 * M * K * E, fcn_head=2.0 * M * E * K, fcn_ln=0.0,
             fcn_mlp=cfg.depth * 2 * (2.0 * M * E * cfg.mlp_ratio * E), fcn_spec=cfg.depth * (dft_w + dft_h + block_mlp))
    f["total"] = sum(f.values())
    return f


def fcn_bytes(cfg: FCNConfig, batch: int = 1) -> dict:
    """Mandatory HBM bytes per step and family for the data flow of csrc/fcn_engine.cu (fp32 token stream x, fp32 LN1
    output u, fp16 LN2 rows, fp16 hidden rows, complex fp32 spectra; weights counted once as fp16 images)."""
    M = batch * cfg.tokens
    E, C, hid = cfg.embed, cfg.n_channels, cfg.mlp_ratio * cfg.embed
    lo, hi = cfg.h_range
    nk, kw, h = hi - lo, cfg.kw, cfg.h
    state = 4.0 * batch * C * cfg.nlat * cfg.nlon
    spec_h = 8.0 * batch * kw * E * (h + nk)                         # one H-DFT pass: read + write
    f = dict(fcn_embed=state + 4.0 * M * E + 2.0 * E * C * 64,
             fcn_head=4.0 * M * E + state + 2.0 * E * C * 64,
             fcn_ln=cfg.depth * (4.0 * M * E * 2 + 4.0 * M * E + 2.0 * M * E),
             fcn_mlp=cfg.depth * (2.0 * M * E + 2.0 * M * hid + 2.0 * 2 * E * hid + 2.0 * M * hid + 4.0 * M * E * 2),
             fcn_spec=cfg.depth * (4.0 * M * E + 8.0 * batch * h * kw * E                 # forward W-DFT
                                   + 2 * spec_h + 2 * 8.0 * batch * nk * kw * E           # H-DFTs, block MLP
                                   + 8.0 * batch * h * kw * E + 4.0 * M * E * 3))          # inverse W-DFT + skips
    f["total"] = sum(f.values())
    return f
