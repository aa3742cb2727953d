"""Differential fuzz: tensor-core Hankel kernels vs the register-tiled direct form (tables = empty) on random shapes with >= 96 tiles,
offline (both delays) and streaming.  One-off robustness check (odd tile counts, partial last tiles, frame counts not a multiple of 4).
Also the half-precision entry points against the fp32 ones (bit-identity) and the host-buffer entries against the device path.
Also the n_band-16 fold / Hankel-16 kernels in their steady state against calls of one tile per CTA.
Arguments: seed, offline cases, host-entry cases, half-precision cases, fold / Hankel-16 cases."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import random, torch
import pqmf_b200 as pq
from pqmf_b200 import _lib
random.seed(int(sys.argv[1]) if len(sys.argv) > 1 else 0)
empty = torch.zeros(0, device="cuda")
worst = {}
for case in range(int(sys.argv[2]) if len(sys.argv) > 2 else 60):
    m = random.choice((4, 8, 16, 16, 32, 64))
    att = random.choice((80, 100, 100, 120))
    try:
        mod = pq.CachedPQMF(att, m).cuda()
    except Exception as e:
        print("ctor", att, m, e); continue
    if mod._tables.numel() == 0: continue
    tiles_per_row = random.choice((1, 1, 2, 3, 5, 9))
    frames = (tiles_per_row * 8192 // m) - random.choice((0, 0, 4, 8, 12, 64, 1, 3)) * random.choice((0, 1))
    frames = max(frames, 8)
    rows = max(1, -(-random.choice((96, 97, 101, 130, 200)) // max(1, -(-frames * m // 8192))))
    x = (0.5 * torch.randn(rows, 1, frames * m, device="cuda")).clamp_(-1, 1)
    f = mod._flags
    for delay in (0, 1):
        y = torch.ops.pqmf_b200.analysis(x, mod.hk, mod._tables, frames, f)
        yd = torch.ops.pqmf_b200.analysis(x, mod.hk, empty, frames, 0)
        o = torch.ops.pqmf_b200.synthesis(yd, mod.hk, mod._tables, delay, f)
        od = torch.ops.pqmf_b200.synthesis(yd, mod.hk, empty, delay, 0)
        ea, es = float((y - yd).abs().max()), float((o - od).abs().max())
        key = (m, att)
        worst[key] = (max(worst.get(key, (0, 0))[0], ea), max(worst.get(key, (0, 0))[1], es))
        lim_s = 1e-5 if m == 64 else 6e-6
        if not (ea <= 3e-6 and es <= lim_s) or not torch.isfinite(o).all():
            print("MISMATCH", dict(m=m, att=att, rows=rows, frames=frames, delay=delay, ea=ea, es=es)); sys.exit(1)
# streaming, n_band 16; every attenuation of tests/test_gpu_stream_banks.py (its banks differ in the streaming plans' history rows and
# pads, and some run the fold kernels or the direct form)
STREAM_ATTENUATIONS = (50, 60, 70, 80, 90, 100, 110, 120, 130, 140)
for case in range(12):
    att = random.choice(STREAM_ATTENUATIONS)
    block = random.choice((512, 1024, 2048, 2304, 4096))
    streams = random.choice((300, 513, 1000)) * (2 if block <= 1024 else 1)
    mod = pq.CachedPQMF(att, 16).cuda(); ref = pq.CachedPQMF(att, 16).cuda(); ref._flags = 0; ref._tables = torch.zeros(0, device="cuda")
    x = (0.5 * torch.randn(streams, 1, 3 * block, device="cuda")).clamp_(-1, 1)
    for i in range(3):
        xb = x[..., i * block:(i + 1) * block].contiguous()
        y, yr = mod.forward_stream(xb), ref.forward_stream(xb)
        o, orf = mod.inverse_stream(yr), ref.inverse_stream(yr)
        ea, es = float((y - yr).abs().max()), float((o - orf).abs().max())
        if not (ea <= 3e-6 and es <= 6e-6):
            print("STREAM MISMATCH", dict(att=att, block=block, streams=streams, i=i, ea=ea, es=es)); sys.exit(1)
# round 2: streaming at n_band 8 / 32, PCM in / out (mono, stereo, down-mix), reconstruct(), process_stream()
for case in range(16):
    m = random.choice((8, 16, 32))
    att = random.choice(STREAM_ATTENUATIONS)
    block = random.choice((512, 1024, 2048, 4096)) * (2 if m == 32 else 1)
    streams = random.choice((300, 400, 1000)) * (2 if block <= 1024 else 1)
    mod = pq.CachedPQMF(att, m).cuda(); ref = pq.CachedPQMF(att, m, fp32=True).cuda()
    x = (0.5 * torch.randn(streams, 1, 3 * block, device="cuda")).clamp_(-1, 1)
    for i in range(3):
        xb = x[..., i * block:(i + 1) * block].contiguous()
        o, y = mod.process_stream(xb)
        yr = ref.forward_stream(xb)
        orf = ref.inverse_stream(y)
        ea, es = float((y - yr).abs().max()), float((o - orf).abs().max())
        if not (ea <= 3e-6 and es <= 8e-6):
            print("STREAM-M MISMATCH", dict(m=m, att=att, block=block, streams=streams, i=i, ea=ea, es=es)); sys.exit(1)
# PCM in / out on every bank the half-precision loop below draws from: bit-equal to the float32 call on the widened rows (synthesis: its
# output quantised) -- the Hankel call where the PCM call runs natively (a bank with tables and >= 96 tiles; synthesis: an unsplit bank),
# the fp32 direct form elsewhere
for case in range(16):
    m = random.choice((4, 8, 16, 16, 32, 64))
    att = random.choice((50, 60, 80, 100, 100, 120, 140))
    c = random.choice((1, 1, 2, 2, 3))
    t = random.choice((8192, 16384, 32768, 40960)) // m * m
    clips = max(1, -(-random.choice((96, 100, 130)) // (c * -(-t // 8192))))
    mod = pq.CachedPQMF(att, m).cuda(); ref = pq.CachedPQMF(att, m, fp32=True).cuda()
    tabled, split = mod._tables.numel() > 0, bool(mod._flags & _lib.PQMF_FLAG_H4_SPLIT)
    pcm = torch.randint(-32768, 32768, (clips, t, c), device="cuda", dtype=torch.int32).to(torch.int16)
    f = pcm.to(torch.float32) / 32768.0
    xf = f.transpose(1, 2).contiguous()
    y = mod.forward_pcm16(pcm)
    if not torch.equal(y, (mod if tabled else ref)(xf)):
        print("PCM ANALYSIS MISMATCH", dict(m=m, att=att, c=c, t=t, clips=clips)); sys.exit(1)
    q = mod.inverse_pcm16(y)
    qr = torch.clamp(torch.round((mod if tabled and not split else ref).inverse(y) * 32768.0), -32768, 32767).to(torch.int16).transpose(1, 2)
    if not torch.equal(q, qr):
        print("PCM SYNTHESIS MISMATCH", dict(m=m, att=att, c=c, t=t, clips=clips)); sys.exit(1)
    if c > 1:  # pcm_sample's down-mix: the fp32 sum in channel order, then / C (a tensor divisor: torch divides by a scalar via its reciprocal)
        acc = f[..., 0].clone()
        for k in range(1, c): acc += f[..., k]
        mono = (acc / torch.full_like(acc, c))[:, None]
        if not torch.equal(mod.forward_pcm16(pcm, True), (mod if tabled and clips * -(-t // 8192) >= 96 else ref)(mono)):
            print("PCM DOWNMIX MISMATCH", dict(m=m, att=att, c=c, t=t, clips=clips)); sys.exit(1)
    if not torch.equal(mod.reconstruct(xf), mod.process(xf)[0]):
        print("RECONSTRUCT MISMATCH", dict(m=m, c=c, t=t, clips=clips)); sys.exit(1)
# host-buffer entry points against the device path: bit-identical whatever the chunk schedule does (tools: PQMF_HOST_CHUNK_MIB=1 makes many chunks)
for case in range(int(sys.argv[3]) if len(sys.argv) > 3 else 12):
    m = random.choice((8, 16, 16, 32))
    c = random.choice((1, 1, 2))
    t = random.choice((2048, 8192, 40960, 65536, 303104, 1 << 20)) // (8 * m) * (8 * m)
    b = random.choice((1, 3, 17, 40, 100, 257))
    if b * c * t > (1 << 27): b = max(1, (1 << 27) // (c * t))
    mod = pq.CachedPQMF(100, m).cuda()
    hk_h, tab_h = mod.hk.cpu().contiguous(), mod._tables.cpu().contiguous()
    L = mod.hk.shape[1]
    if random.random() < 0.5:
        x = (0.5 * torch.randn(b * c, 1, t)).clamp_(-1, 1)
        hx = x.pin_memory(); ho = torch.empty(b * c, t).pin_memory(); hy = torch.empty(b * c, m, t // m).pin_memory()
        rc = _lib.cabi.pqmf_roundtrip_host_f32(hx.data_ptr(), hy.data_ptr(), ho.data_ptr(), hk_h.data_ptr(), tab_h.data_ptr(), b * c, t, m, L, 1, int(mod._flags), 0)
        y = mod(x.cuda()); o = mod.inverse(y)
        ok = rc == 0 and torch.equal(hy, y.cpu()) and torch.equal(ho, o.cpu()[:, 0])
    else:
        pcm = torch.randint(-32768, 32768, (b, t, c), dtype=torch.int32).to(torch.int16)
        hp = pcm.pin_memory(); ho = torch.empty_like(hp).pin_memory(); hy = torch.empty(b * c, m, t // m).pin_memory()
        rc = _lib.cabi.pqmf_roundtrip_host_pcm16(hp.data_ptr(), hy.data_ptr(), ho.data_ptr(), hk_h.data_ptr(), tab_h.data_ptr(), b, t, c, m, L, 1, int(mod._flags), 0)
        y = mod.forward_pcm16(pcm.cuda()); o = mod.inverse_pcm16(y)
        ok = rc == 0 and torch.equal(hy, y.cpu().reshape(hy.shape)) and torch.equal(ho, o.cpu())
    if not ok:
        print("HOST ENTRY MISMATCH", dict(m=m, c=c, t=t, b=b, rc=rc)); sys.exit(1)
# half-precision I/O: bit-identical to the fp32 call on the widened input, rounded -- on random shapes around the boundary between the
# native half-precision kernels and the staged path (T % 8, frames % 4, tile count near 96, base pointer offset), on every bank the
# half-precision kernels serve (attenuation 50 .. 140), and from one tile per CTA up to ~10 (the steady state of the persistent loop)
for case in range(int(sys.argv[4]) if len(sys.argv) > 4 else 40):
    m = random.choice((4, 8, 16, 16, 32, 64))
    att = random.choice((50, 60, 80, 100, 100, 120, 140))
    dt = random.choice((torch.float16, torch.bfloat16))
    cls = random.choice((pq.PQMF, pq.CachedPQMF))
    mod = cls(att, m, exact=random.random() < 0.25).cuda()
    tpr = random.choice((1, 2, 3, 8))
    t = tpr * 8192 - random.choice((0, 0, 8 * m, 4 * m, 2 * m, m, 4, 3))
    if cls is pq.PQMF: t -= t % m  # polyphase: whole frames
    tiles = random.choice((96, 96, 97, 149, 297, 601, 1221, 1480))
    rows = max(1, -(-tiles // -(-t // 8192)) + random.choice((-1, 0, 0, 1)))
    offset = random.choice((0, 0, 0, 1, 8))
    flat = (0.5 * torch.randn(rows * t + offset, device="cuda")).clamp_(-1, 1).to(dt)
    x = flat[offset:offset + rows * t].view(rows, 1, t)
    y = mod(x)
    o = mod.inverse(y)
    if not (torch.equal(y.view(torch.int16), mod(x.float()).to(dt).view(torch.int16)) and
            torch.equal(o.view(torch.int16), mod.inverse(y.float()).to(dt).view(torch.int16)) and y.dtype == dt and o.dtype == dt):
        print("HALF MISMATCH", dict(m=m, att=att, dtype=str(dt), cls=cls.__name__, rows=rows, t=t, offset=offset)); sys.exit(1)
# n_band 16 fold / Hankel-16 kernels (exact on / off) in the steady state of their persistent loops: lockstep streaming with blocks that
# are not a multiple of 256 samples (the Hankel-4 streaming kernels refuse them) at 1000 - 5000 streams, and offline batches whose signal
# sits 16 bytes past a 32-byte boundary and sub-bands 4 bytes past a 16-byte one (the Hankel-4 kernels refuse them).  Every row bit-equal
# to calls of at most one tile per CTA (groups of 16 streams; offline row chunks of at most 2 x SMs tiles in any family) with the
# family's forced flags -- a tile's output does not depend on which CTA runs it at which iteration.
n_sm = torch.cuda.get_device_properties(0).multi_processor_count
for case in range(int(sys.argv[5]) if len(sys.argv) > 5 else 12):
    att = random.choice((80, 100, 110, 120, 130))
    exact = random.random() < 0.5
    cls = random.choice((pq.PQMF, pq.CachedPQMF))
    mod = cls(att, 16, exact=exact).cuda()
    f = mod._flags
    forced = f | _lib.PQMF_FLAG_FOLD | (_lib.PQMF_FLAG_NO_FOLD if exact else 0)
    hk, tab = mod.hk, mod._tables
    if cls is pq.CachedPQMF and random.random() < 0.5:
        streams = random.randint(1000, 5000)
        plan = [random.choice((480, 960, 1920, 4800, 496, 48, 16)) for _ in range(4)]
        for k, T in enumerate(plan):
            x = (0.5 * torch.randn(streams, 1, T, device="cuda")).clamp_(-1, 1)
            xs_in = mod._x_state[mod._x_slot].clone() if k else torch.zeros(streams, 512, device="cuda")
            ss_in = mod._s_state[mod._s_slot].clone() if k else torch.zeros(streams, 512, device="cuda")
            pin, pout = mod._frames_in % 2, mod._frames_out % 2
            out, y = mod.process_stream(x)
            for g in range(0, streams, 16):
                xi, si = xs_in[g:g + 16], ss_in[g:g + 16]
                o_r, y_r = torch.ops.pqmf_b200.stream_step(x[g:g + 16], hk, tab, xi, torch.empty_like(xi), si, torch.empty_like(si), pin, pout, forced)
                if not (torch.equal(y[g:g + 16], y_r) and torch.equal(out[g:g + 16], o_r)):
                    print("FOLD STREAM MISMATCH", dict(att=att, exact=exact, streams=streams, plan=plan, k=k, group=g)); sys.exit(1)
    else:
        rows, F = random.randint(100, 1500), random.randint(1, 2048)
        delay = 1 if cls is pq.CachedPQMF else 0
        x0 = (0.5 * torch.randn(rows, 1, 16 * F, device="cuda")).clamp_(-1, 1)
        x = torch.empty(x0.numel() + 16, device="cuda")[4:4 + x0.numel()].view(x0.shape).copy_(x0)
        y = mod(x)
        s = torch.empty(y.numel() + 16, device="cuda")[1:1 + y.numel()].view(y.shape).copy_(y)
        out = mod.inverse(s)
        per = max(1, 2 * n_sm // -(-F // 64))  # rows per reference call: at most one tile per CTA in every family and direction
        y_r = torch.cat([torch.ops.pqmf_b200.analysis(x0[i:i + per].clone(), hk, tab, F, forced) for i in range(0, rows, per)])
        o_r = torch.cat([torch.ops.pqmf_b200.synthesis(y[i:i + per].clone(), hk, tab, delay, forced) for i in range(0, rows, per)])
        if not (torch.equal(y, y_r) and torch.equal(out, o_r)):
            print("FOLD OFFLINE MISMATCH", dict(att=att, exact=exact, cls=cls.__name__, rows=rows, F=F)); sys.exit(1)
print("fuzz ok; worst |hankel - direct| per (n_band, attenuation):", {k: (f"{v[0]:.1e}", f"{v[1]:.1e}") for k, v in sorted(worst.items())})
