"""numpy restatement of the tracer-particle model of latticeurbanwind_b200/csrc/lbm_particles.cuh (luw_particles_*), written from its definition, not from
the kernel: float64 positions in lattice coordinates (cell centres at integers), float32 trilinear velocity from the 8 cells around a particle, explicit Euler
plus a uniform random walk from Philox4x64-10, periodic wrap, open faces (LEFT), wall modes (reject / DEPOSITED), box emitters (BURIED in solids) and
concentration bins. Every float32 / float64 operation below is one IEEE operation rounded to nearest, in the order the definition gives.

Cell velocities are the caller's: the u that update_fields + a read gives at each cell (the C oracle's update_fields on a copy of the fields, or the stored
u where update_fields leaves it), float32 [3, N] in the dense order n = x + (y + z*Ny)*Nx."""
import numpy as np

FREE, ACTIVE, DEPOSITED, LEFT, BURIED = 0, 1, 2, 3, 4
_M0, _M1 = np.uint64(0xD2E7470EE14C6C93), np.uint64(0xCA5A826395121157)
_W0, _W1 = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xBB67AE8584CAA73B)
_LO32, _S32 = np.uint64(0xFFFFFFFF), np.uint64(32)


def _mulhilo(a, b):
    """-> (high, low) 64-bit words of the 128-bit products a*b (uint64 arrays)"""
    al, ah, bl, bh = a & _LO32, a >> _S32, b & _LO32, b >> _S32
    ll, lh, hl, hh = al * bl, al * bh, ah * bl, ah * bh
    mid = (ll >> _S32) + (lh & _LO32) + (hl & _LO32)
    return hh + (lh >> _S32) + (hl >> _S32) + (mid >> _S32), a * b


def philox4x64_10(counter, key):
    """Philox4x64-10 blocks for counters uint64 [n, 4] and keys uint64 [n, 2] (or [2]) -> uint64 [n, 4]. Equals np.random.Philox(counter=c-1, key=k).random_raw(4)
    (numpy increments its counter before it produces a block)."""
    x = np.array(counter, np.uint64).reshape(-1, 4).T.copy()
    k = np.broadcast_to(np.asarray(key, np.uint64).reshape(-1, 2), (x.shape[1], 2)).T.copy()
    with np.errstate(over="ignore"):
        for _ in range(10):
            hi0, lo0 = _mulhilo(_M0, x[0])
            hi1, lo1 = _mulhilo(_M1, x[2])
            x = np.stack([hi1 ^ x[1] ^ k[0], lo1, hi0 ^ x[3] ^ k[1], lo0])
            k = np.stack([k[0] + _W0, k[1] + _W1])
    return x.T.copy()


def _sym(r):
    """2U - 1 with U = (r >> 11) * 2^-53"""
    return 2.0 * ((r >> np.uint64(11)).astype(np.float64) * 2.0 ** -53) - 1.0


def _wrap(q, N):
    q = q.copy()
    m = ~((q >= 0.0) & (q < N))
    with np.errstate(invalid="ignore"):
        r = q[m] - np.floor(q[m] / N) * N
        r = np.where(r < 0.0, r + N, r)
        r = np.where(r >= N, r - N, r)
    q[m] = r
    return q


def _nearest(q, N):
    k = np.floor(q + 0.5).astype(np.int64)
    return np.where(k >= N, k - N, k)


class ParticleRing:
    """One luw_particles object: shape (Nx, Ny, Nz), emitters [E, 6] (cx cy cz hx hy hz), periodic_mask bits x y z, wall_mode 0 / 1, seed, bin_size (bx, by, bz)."""

    def __init__(self, shape, capacity, emitters, periodic_mask=0, wall_mode=0, seed=0, bin_size=(1, 1, 1)):
        self.shape = tuple(int(v) for v in shape)
        self.capacity = int(capacity)
        self.emitters = np.asarray(emitters, np.float64).reshape(-1, 6)
        self.periodic = [bool((int(periodic_mask) >> a) & 1) for a in range(3)]
        self.wall_mode, self.seed = int(wall_mode), np.uint64(seed)
        self.b = tuple(int(v) for v in bin_size)
        self.B = tuple((n + b - 1) // b for n, b in zip(self.shape, self.b))
        self.p = np.zeros((3, self.capacity), np.float64)
        self.state = np.zeros(self.capacity, np.uint8)
        self.emitter = np.zeros(self.capacity, np.uint32)
        self.release = np.zeros(self.capacity, np.uint64)
        self.bins = np.zeros(self.B[::-1], np.uint32)
        self.head = self.emit_calls = self.advance_calls = self.samples = 0

    def _random(self, slots, call, stream):
        ctr = np.zeros((slots.size, 4), np.uint64)
        ctr[:, 0], ctr[:, 1], ctr[:, 2] = slots, call, stream
        return philox4x64_10(ctr, [self.seed, 0])

    def _solid(self, flags, q):
        Nx, Ny, Nz = self.shape
        n = _nearest(q[0], Nx) + (_nearest(q[1], Ny) + _nearest(q[2], Nz) * Ny) * Nx
        return (flags[n] & 0x03) == 0x01

    def emit(self, flags, t, per_emitter):
        total = self.emitters.shape[0] * int(per_emitter)
        assert total <= self.capacity
        if total:
            i = np.arange(total, dtype=np.uint64)
            slots = (np.uint64(self.head) + i) % np.uint64(self.capacity)
            e = (i // np.uint64(per_emitter)).astype(np.int64)
            r = self._random(slots, self.emit_calls, 1)
            q = np.empty((3, total), np.float64)
            for a in range(3):
                q[a] = self.emitters[e, a] + self.emitters[e, 3 + a] * _sym(r[:, a])
                if self.periodic[a]:
                    q[a] = _wrap(q[a], float(self.shape[a]))
            s = slots.astype(np.int64)
            self.p[:, s] = q
            self.state[s] = np.where(self._solid(flags, q), BURIED, ACTIVE)
            self.emitter[s] = e
            self.release[s] = t
            self.head = (self.head + total) % self.capacity
        self.emit_calls += 1

    def velocity(self, ucell, p):
        """float32 [3, n]: trilinear interpolation of the cell velocities ucell [3, N] at the positions p [3, n]"""
        lo, hi, f = [], [], []
        for a in range(3):
            N = self.shape[a]
            x0 = np.floor(p[a]).astype(np.int64)
            if not self.periodic[a]:
                x0 = np.minimum(x0, N - 2)
            x1 = x0 + 1
            if self.periodic[a]:
                x1 = np.where(x1 == N, 0, x1)
            lo.append(x0); hi.append(x1); f.append((p[a] - x0).astype(np.float32))
        Nx, Ny, _ = self.shape
        one = np.float32(1.0)

        def lerp(a, b, w):
            return a * (one - w) + b * w

        def cell(ix, iy, iz):
            return ucell[:, ix + (iy + iz * Ny) * Nx]
        edge = {(y, z): lerp(cell(lo[0], (lo, hi)[y][1], (lo, hi)[z][2]), cell(hi[0], (lo, hi)[y][1], (lo, hi)[z][2]), f[0]) for y in (0, 1) for z in (0, 1)}
        face = [lerp(edge[(0, z)], edge[(1, z)], f[1]) for z in (0, 1)]
        return lerp(face[0], face[1], f[2])

    def advance(self, ucell, flags, dt=1.0, sigma=0.0):
        s = np.nonzero(self.state == ACTIVE)[0]
        if s.size:
            p = self.p[:, s]
            u = self.velocity(np.asarray(ucell, np.float32).reshape(3, -1), p)
            r = self._random(s.astype(np.uint64), self.advance_calls, 0)
            amp = np.float64(sigma) * np.sqrt(3.0)
            dt64 = np.float64(np.float32(dt))
            q = np.empty_like(p)
            left = np.zeros(s.size, bool)
            for a in range(3):
                q[a] = p[a] + u[a].astype(np.float64) * dt64 + amp * _sym(r[:, a])
                N = float(self.shape[a])
                if self.periodic[a]:
                    q[a] = _wrap(q[a], N)
                    left |= ~((q[a] >= 0.0) & (q[a] < N))
                else:
                    left |= ~((q[a] >= 0.0) & (q[a] <= N - 1.0))
            solid = np.zeros(s.size, bool)
            solid[~left] = self._solid(flags, q[:, ~left])
            move = left | ~solid | (self.wall_mode == 1)
            self.p[:, s[move]] = q[:, move]
            self.state[s[left]] = LEFT
            self.state[s[~left & solid & (self.wall_mode == 1)]] = DEPOSITED
        self.advance_calls += 1

    def count(self):
        s = self.state == ACTIVE
        idx = [_nearest(self.p[a, s], self.shape[a]) // self.b[a] for a in range(3)]
        np.add.at(self.bins, (idx[2], idx[1], idx[0]), np.uint32(1))
        self.samples += 1

    def reset_bins(self):
        self.bins[:] = 0
        self.samples = 0
