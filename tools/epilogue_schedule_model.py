"""CPU restatement of the lean GEMM epilogue's bookkeeping (csrc/gemm_tcgen05.cu, `kEpi != E_GENERIC`) — verification aid.

The device code replaces divisions, modulo ring indices and a leader warp by incremental counters; this model runs the SAME updates for
both epilogue groups of one CTA and checks them against the straightforward definitions:
  * the division-free tile iterator visits exactly the units u = first + i * stride -> (u // n_tiles, u % n_tiles);
  * every 32-column chunk of every tile is owned by exactly one group (plain: alternate chunks, the odd one alternating from tile to
    tile; GEGLU: alternate (value, gate) chunk pairs);
  * the residual prefetch cursor — advanced independently, two loads ahead — produces exactly the (tile, chunk) sequence the group
    consumes, in the same buffer order;
  * with kOB output staging buffers, the store that last read a buffer was issued kOB chunks earlier by warp (turn - kOB) & 3, and that
    warp's wait sits in the iteration before the buffer is staged again ((turn + 5 - kOB) & 3 == the issuer of chunk n - (kOB - 1));
  * block-shaped conv tiles (box_h x box_w pixels of one frame, or whole frames): the tile origin and per-row pixel the epilogue
    derives cover every output pixel exactly once, and each tile's clipped store box holds exactly its valid rows.
"""
from __future__ import annotations


def group_schedule(eg: int, first_unit: int, stride: int, n_tiles: int, num_units: int, N: int, BN: int, geglu: bool, k_ob: int = 2):
    """what epilogue group `eg` of one CTA does: list of (m_unit, n_tile, chunk, out_buffer, issuing_warp, waits_for_chunk_index)"""
    step, log = (4, 2) if geglu else (2, 1)
    dm, dn = stride // n_tiles, stride % n_tiles
    mu_count = num_units // n_tiles
    mu, n_tile = first_unit // n_tiles, first_unit % n_tiles
    full_chunks = BN // 32

    def chunks_of(n):
        nc = (N - n * BN + 31) >> 5
        return min(nc, full_chunks)

    out, ob, turn, par, idx = [], 0, 0, 0, 0
    while mu < mu_count:
        nchunks = chunks_of(n_tile)
        first = 2 * eg if geglu else (eg ^ par)
        n_own = (nchunks - first + step - 1) >> log if nchunks > first else 0
        c = first
        for _ in range(n_own):
            waiter = (turn + 5 - k_ob) & 3           # the warp that confirms a finished store read in this iteration
            out.append(dict(mu=mu, n=n_tile, c=c, ob=ob, turn=turn, waiter=waiter, idx=idx))
            ob = 0 if ob == k_ob - 1 else ob + 1
            turn = (turn + 1) & 3
            c += step
            idx += 1
        n_tile += dn
        mu += dm
        if n_tile >= n_tiles:
            n_tile -= n_tiles
            mu += 1
        par ^= 1
    return out


def prefetch_sequence(eg: int, first_unit: int, stride: int, n_tiles: int, num_units: int, N: int, BN: int, geglu: bool):
    """the residual prefetcher's own cursor (prefetch_one of the lean epilogue): (m_unit, n_tile, chunk, res_buffer) per load"""
    step = 4 if geglu else 2
    dm, dn = stride // n_tiles, stride % n_tiles
    mu_count = num_units // n_tiles
    pf_mu, pf_n = first_unit // n_tiles, first_unit % n_tiles
    full_chunks = BN // 32
    chunks_of = lambda n: min((N - n * BN + 31) >> 5, full_chunks)
    pf_c, pf_par, pf_buf, out = (2 * eg if geglu else eg), 0, 0, []
    while True:
        while pf_mu < mu_count and pf_c >= chunks_of(pf_n):
            pf_n += dn
            pf_mu += dm
            if pf_n >= n_tiles:
                pf_n -= n_tiles
                pf_mu += 1
            pf_par ^= 1
            pf_c = 2 * eg if geglu else (eg ^ pf_par)
        if pf_mu >= mu_count:
            return out
        out.append((pf_mu, pf_n, pf_c, pf_buf))
        pf_buf ^= 1
        pf_c += step


def check(first_unit, stride, m_units, n_tiles, N, BN, geglu, k_ob=2):
    num_units = m_units * n_tiles
    units = [(u // n_tiles, u % n_tiles) for u in range(first_unit, num_units, stride)]
    sched = [group_schedule(eg, first_unit, stride, n_tiles, num_units, N, BN, geglu, k_ob) for eg in (0, 1)]
    # tiles visited = the CTA's units, in order, by both groups
    for eg in (0, 1):
        seen = []
        for e in sched[eg]:
            if not seen or seen[-1] != (e["mu"], e["n"]):
                seen.append((e["mu"], e["n"]))
        assert [t for t in units if t in seen] == seen, (eg, seen[:4], units[:4])
    # chunk ownership: each chunk (GEGLU: each chunk pair) of every tile exactly once
    for ti, (mu, n) in enumerate(units):
        nchunks = min((N - n * BN + 31) >> 5, BN // 32)
        owned = sorted((e["c"], eg) for eg in (0, 1) for e in sched[eg] if (e["mu"], e["n"]) == (mu, n))
        want = list(range(0, nchunks, 2)) if geglu else list(range(nchunks))
        assert [c for c, _ in owned] == want, (mu, n, owned, want)
        if not geglu and nchunks % 2 == 1 and nchunks > 1:  # the group with the extra chunk alternates from tile to tile
            extra = max((0, 1), key=lambda g: sum(1 for c, eg in owned if eg == g))
            assert extra == (ti & 1), (ti, owned)
    # residual prefetcher == consumption order, buffers alternate
    for eg in (0, 1):
        pf = prefetch_sequence(eg, first_unit, stride, n_tiles, num_units, N, BN, geglu)
        assert [(a, b, c) for a, b, c, _ in pf] == [(e["mu"], e["n"], e["c"]) for e in sched[eg]]
        assert [buf for *_, buf in pf] == [i & 1 for i in range(len(pf))]
    # output ring: buffer of chunk i was last the source of the store of chunk i - kOB (issued by warp (i - kOB) & 3); its read is
    # confirmed in iteration i - 1 by `waiter`, which must be that issuer
    for eg in (0, 1):
        s = sched[eg]
        for i, e in enumerate(s):
            assert e["ob"] == i % k_ob and e["turn"] == i % 4
            if i >= 1 and i - k_ob >= 0:
                assert s[i - 1]["waiter"] == s[i - k_ob]["turn"], (i, s[i - 1], s[i - k_ob])
    return sum(len(x) for x in sched)


def conv_tile_origin(plan, W, m_tile):
    """conv_tile_origin of the device code: first output pixel (n0, y0, x0) of a conv tile.  `plan` = (box_w, box_h,
    frames_per_tile, tiles_per_frame, m_tiles) as av2v_conv3x3_plan returns it."""
    box_w, box_h, fpt, tpf, _ = plan
    if fpt > 1:
        return m_tile * fpt, 0, 0
    x_tiles = -(-W // box_w)
    n0 = m_tile // tpf
    yb, xb = divmod(m_tile - n0 * tpf, x_tiles)
    return n0, yb * box_h, xb * box_w


def block_tile_pixels(plan, NF, H, W, m_tile):
    """the output pixels the epilogue writes for accumulator rows r = 0..127 of a block-shaped tile: {r: (n, y, x)} for the
    rows it treats as valid (row-bias index, and the rows the clipped TMA store box keeps)"""
    box_w, box_h, fpt, _, _ = plan
    n0, y0, x0 = conv_tile_origin(plan, W, m_tile)
    out = {}
    for r in range(128):
        bz, rr = divmod(r, box_w * box_h)
        by, bx = divmod(rr, box_w)
        n, y, x = n0 + bz, y0 + by, x0 + bx
        if bz < fpt and x < W and y < H and n < NF:
            out[r] = (n, y, x)
    return out


def check_block_tiles(plan, NF, H, W, pair=False):
    """every output pixel is written by exactly one (tile, row); a tile's store box {box_w, box_h, frames} at its origin, clipped
    to the image, holds exactly its valid rows (so a box never reaches into the next frame or row); rows are in the A box's
    shared-memory order.  pair: the tile schedule of CTA pairs (2 mu + rank) including the phantom tile of an odd m_tiles."""
    box_w, box_h, fpt, tpf, m_tiles = plan
    assert box_w * box_h * fpt <= 128 and max(box_w, box_h, fpt) <= 256
    seen = {}
    tiles = range(2 * (-(-m_tiles // 2))) if pair else range(m_tiles)
    for m in tiles:
        px = block_tile_pixels(plan, NF, H, W, m)
        if m >= m_tiles:
            assert not px, f"phantom pair tile {m} writes {len(px)} pixels"
            continue
        n0, y0, x0 = conv_tile_origin(plan, W, m)
        assert n0 < NF and y0 < H and x0 < W, (m, n0, y0, x0)
        box = {(n, y, x) for n in range(n0, min(n0 + fpt, NF)) for y in range(y0, min(y0 + box_h, H))
               for x in range(x0, min(x0 + box_w, W))}
        assert set(px.values()) == box, (m, len(px), len(box))
        for r, pix in px.items():
            assert pix not in seen, f"pixel {pix} written by tiles {seen[pix]} and {m}"
            seen[pix] = m
    assert len(seen) == NF * H * W, (len(seen), NF * H * W)
    return len(seen)


if __name__ == "__main__":
    total = 0
    for BN, N, geglu in ((160, 960, False), (160, 320, False), (256, 2560, True), (128, 320, False), (64, 200, False), (256, 1280, False), (128, 1280, True)):
        n_tiles = (N + BN - 1) // BN
        for first, stride, m_units in ((0, 148, 1536), (147, 148, 1536), (3, 7, 40), (5, 74, 193)):
            for k_ob in (2, 3):
                total += check(first, stride, m_units, n_tiles, N, BN, geglu, k_ob)
    print(f"lean epilogue bookkeeping: {total} chunk visits checked")
    # block tiles of 1280 x 704 (latent 160 x 88 and its levels): plans as av2v_conv3x3_plan returns them
    px = sum(check_block_tiles(plan, 3, H, W, pair=True) for plan, H, W in (((32, 4, 1, 110, 330), 88, 160), ((16, 8, 1, 30, 90), 44, 80),
                                                                             ((40, 3, 1, 8, 24), 22, 40), ((20, 6, 1, 2, 6), 11, 20)))
    print(f"block conv tiles: {px} output pixels covered exactly once")
