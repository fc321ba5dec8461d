"""Operand bytes into the SMs (L2 -> shared memory, by TMA) and tcgen05 MMA count of ONE DiffNet layer in the fused layer kernel
(bisinger_b200/csrc/diffnet_layer.cuh), computed from the shapes -- no GPU involved.

Two tilings of the rows:
  item     each item's rows in 256-row tiles (tile m -> item m / ceil(T / 256)), one 128-row half per CTA of the pair;
  slab     128-row slabs numbered across the batch, pair tile u = slabs 2u and 2u + 1 (the kernel's tiling).
A third row counts the halo slabs of a pair tile once for both gate ops (both channel halves) instead of once per gate op, a
variant that was measured and not kept (DESIGN.md §9).

Per CTA and pair tile: gate ops 2 x (12 fp16 + 6 e5m2 weight tiles of 128 rows x 128 B, 6 halo boxes of a_rows x 128 B),
residual op 8 weight tiles + 4 z boxes of 128 x 128 B, epilogue boxes 2 x 16 cp + 8 conv-input boxes of 128 rows x 64 B.
Rows a TMA box reads outside [0, T) of its item (halo rows before row 0 or past T, the rows of a missing slab) are zero-filled
by the TMA unit and counted as moving no bytes; weight tiles are loaded in full by every CTA of a busy pair.

    python tools/layer_bytes.py                      # cfg3: B = 32, T = 1875, 20 layers, dilation cycle 4
    python tools/layer_bytes.py --B 1 --T 300 --a-stages 6 --w-stages 4 --e-stages 6
"""
import argparse

C = 256
TILE_M = 128
A_ROWS = 144                  # halo box rows (128 + 2 x the largest dilation, rounded to 8)
W_TILE = 128 * 128            # weight tile: 128 N rows x 128 B
E_BOX = 128 * 16 * 4          # epilogue box: 128 rows x 64 B
MMA_GATE16, MMA_GATE8, MMA_RES = 4 * 3 * 4, 2 * 3 * 4, 4 * 2 * 4   # per op and pair tile (K = 16 / K = 32 / K = 16 instructions)


def rows_in(t0, n, T):
    return max(0, min(t0 + n, T) - max(t0, 0))


def cta_bytes(t0, T, dil, live, shared_halo):
    """bytes one CTA takes in for one pair tile; t0: first row of its 128 in the item, live: the CTA has an item (not a missing slab)"""
    w = 2 * (12 + 6) * W_TILE + 8 * W_TILE
    if not live:
        return {"weights": w, "halo": 0, "z": 0, "cp": 0, "xe": 0}
    own = rows_in(t0, TILE_M, T)
    halo = 6 * rows_in(t0 - dil, A_ROWS, T) * 128 * (1 if shared_halo else 2)
    return {"weights": w, "halo": halo, "z": 4 * own * 128, "cp": 2 * 16 * own * 64, "xe": 8 * own * 64}


def layer(B, T, dil, tiling, shared_halo):
    """(bytes by operand, pair tiles, MMA instructions) of one layer"""
    ctas = []   # (t0, live) of every CTA-tile
    if tiling == "item":
        for b in range(B):
            for m in range((T + 2 * TILE_M - 1) // (2 * TILE_M)):
                ctas += [(m * 2 * TILE_M, True), (m * 2 * TILE_M + TILE_M, True)]
    else:
        S = (T + TILE_M - 1) // TILE_M
        ctas = [(s * TILE_M, True) for b in range(B) for s in range(S)]
        if len(ctas) % 2:
            ctas.append((0, False))
    tot = {}
    for t0, live in ctas:
        for k, v in cta_bytes(t0, T, dil, live, shared_halo).items():
            tot[k] = tot.get(k, 0) + v
    pairs = len(ctas) // 2
    return tot, pairs, pairs * (2 * (MMA_GATE16 + MMA_GATE8) + MMA_RES)


def smem_plan(a_stages, w_stages, e_stages):
    """LayerSmem::kTotal for these ring depths (diffnet_layer.cuh)"""
    return a_stages * A_ROWS * 128 + w_stages * W_TILE + e_stages * E_BOX + 2 * 256 * 4 + 512 + 1024


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--B", type=int, default=32)
    ap.add_argument("--T", type=int, default=1875)
    ap.add_argument("--layers", type=int, default=20)
    ap.add_argument("--dilation-cycle", type=int, default=4)
    ap.add_argument("--pairs", type=int, default=74, help="CTA pairs of the persistent grid (B200: 148 SMs)")
    ap.add_argument("--a-stages", type=int, default=3)
    ap.add_argument("--w-stages", type=int, default=6)
    ap.add_argument("--e-stages", type=int, default=9)
    a = ap.parse_args()
    dils = [2 ** (l % a.dilation_cycle) for l in range(a.layers)]
    assert max(dils) <= (A_ROWS - TILE_M) // 2, "dilation too long for the halo box"
    print(f"B = {a.B}, T = {a.T}, {a.layers} layers, dilations {sorted(set(dils))}; per layer (mean over the layers):")
    base = None
    for tiling, shared in (("item", False), ("slab", False), ("slab", True)):
        per = [layer(a.B, a.T, d, tiling, shared) for d in dils]
        tot = {k: sum(p[0][k] for p in per) / len(per) for k in per[0][0]}
        mb = sum(tot.values()) / 1e6
        pairs, mmas = per[0][1], per[0][2]
        base = base or (mb, mmas)
        parts = ", ".join(f"{k} {v / 1e6:.1f}" for k, v in tot.items())
        name = f"{tiling}{' + shared halo' if shared else ''}"
        print(f"  {name:19s} {mb:7.1f} MB ({mb / base[0] - 1:+.1%})  [{parts}]  pair tiles {pairs} "
              f"({pairs / a.pairs:.2f} per pair)  MMAs {mmas} ({mmas / base[1] - 1:+.1%})")
    s = smem_plan(a.a_stages, a.w_stages, a.e_stages)
    print(f"shared memory with rings A {a.a_stages} / W {a.w_stages} / E {a.e_stages}: {s} B ({s / 1024:.1f} KB of 227 KB)"
          f"{'' if s <= 227 * 1024 else '  -- DOES NOT FIT'}")


if __name__ == "__main__":
    main()
