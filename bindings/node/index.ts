// TypeScript face of the engine: the reference's API names on top of the N-API addon (addon.c).
// NOT BUILT OR RUN IN THIS REPOSITORY'S IMAGE (no Node.js); the Python host layer montgomery_b200/api.py is the
// tested mirror of the same interface.  Shapes follow the reference:
//   Weierstraß.create(params) -> { Parallel: { pointsFromBytes, randomPointsFast, msm, msmUnsafe, msmProjective } }
//     (src/parallel.ts:40-176), msm(scalars, points, N, verbose?, {c?}) -> {result, log} (src/msm-batched-affine.ts:69-78,339)
//   compute_msm(points, scalars) -> {x, y}      (scripts/zprize23/submission-bls377.ts:20-65)
// Difference that a caller sees: `scalarPtr` / `pointPtr` are not offsets into wasm memory but a Uint8Array of
// 32-byte little-endian scalars and a handle to points resident in GPU memory.
// eslint-disable-next-line @typescript-eslint/no-var-requires
const addon = require("./build/Release/montgomery_b200.node");

export enum Curve { BLS12_377_G1 = 0, PALLAS = 1, ED_ON_BLS12_377 = 2, BLS12_381_G1 = 3 }
const coordBytes: Record<Curve, number> = { 0: 48, 1: 32, 2: 32, 3: 48 };

export type MsmResult = { result: { x: bigint; y: bigint; isZero: boolean }; log: Record<string, number> };
export type Points = { readonly n: number };                    // the "pointPtr": points live in HBM inside the engine

const fromLE = (b: Uint8Array) => b.reduceRight((acc, v) => (acc << 8n) | BigInt(v), 0n);

export function create(curve: Curve, { device = 0, maxPoints = 1 << 20 } = {}) {
  const ctx = addon.create(curve, device, maxPoints);
  const cb = coordBytes[curve];
  async function run(scalars: Uint8Array, points: Points, N: number, c = 0, projective = 0): Promise<MsmResult> {
    if (N > points.n) throw Error(`msm: N = ${N} exceeds the ${points.n} points held`);
    const { xy, isZero, log } = await addon.msm(ctx, scalars, N, c, projective);
    return { result: { x: fromLE(xy.subarray(0, cb)), y: fromLE(xy.subarray(cb, 2 * cb)), isZero }, log };
  }
  const Parallel = {
    // src/parallel.ts:97-116 / :209-232.  check: every point is checked on the GPU (canonical, on the curve, in the
    // prime-order subgroup: isOnCurve / isInSubgroup); an invalid one throws "<count> invalid points; the first is point
    // <i>: <reason>" and the engine holds no points.
    pointsFromBytes(bytes: Uint8Array, { check = false } = {}): Points {
      const n = bytes.length / (2 * cb);
      addon.setPoints(ctx, bytes, n, check ? 1 : 0);
      return { n };
    },
    randomPointsFast(n: number, seed = 0x6d6f6e74): Points {    // src/curve-random.ts:24-92
      addon.randomPoints(ctx, seed, n);
      return { n };
    },
    msm: (scalars: Uint8Array, points: Points, N: number, _verbose = false, { c = 0 } = {}) => run(scalars, points, N, c),
    // every addition of the engine is complete, so the "unsafe" variant is the same call
    msmUnsafe: (scalars: Uint8Array, points: Points, N: number, _verbose = false, { c = 0 } = {}) => run(scalars, points, N, c),
    msmProjective: (scalars: Uint8Array, points: Points, N: number, { c = 0 } = {}) => run(scalars, points, N, c, 1),
    // extension: start uploading the scalars of the NEXT msm call while the current one runs (mgb_msm_prefetch); pass the
    // same Uint8Array and N to msm afterwards and keep it unchanged until that call resolves
    prefetchScalars(scalars: Uint8Array, N: number): void { addon.prefetch(ctx, scalars, N); },
  };
  return { Parallel };
}

// Several GPUs behind the same `Parallel` shape.  The reference scales by `startThreads(n)` and a per-thread split of the
// inputs (src/threads/threads.ts:354-359, msm-batched-affine.ts:311-320); here `devices` plays the role of the thread count:
// the library splits the point set contiguously over the GPUs, each computes a partial sum, one NCCL all-gather and a
// point addition combine them (mgb_multi_*: contexts and communicators live inside the library, one Node process).
export function createSharded(curve: Curve, { devices = [0], maxPointsPerDevice = 1 << 21 } = {}) {
  const mctx = addon.createMulti(curve, Int32Array.from(devices), maxPointsPerDevice);
  const cb = coordBytes[curve];
  async function run(scalars: Uint8Array, points: Points, N: number, c = 0): Promise<MsmResult> {
    if (N > points.n) throw Error(`msm: N = ${N} exceeds the ${points.n} points held`);
    const { xy, isZero, log } = await addon.msmSharded(mctx, scalars, N, c);
    return { result: { x: fromLE(xy.subarray(0, cb)), y: fromLE(xy.subarray(cb, 2 * cb)), isZero }, log };
  }
  const Parallel = {
    pointsFromBytes(bytes: Uint8Array): Points { const n = bytes.length / (2 * cb); addon.setPointsMulti(mctx, bytes, n); return { n }; },
    randomPointsFast(n: number, seed = 0x6d6f6e74): Points { addon.randomPointsMulti(mctx, seed, n); return { n }; },
    msm: (scalars: Uint8Array, points: Points, N: number, _verbose = false, { c = 0 } = {}) => run(scalars, points, N, c),
    msmUnsafe: (scalars: Uint8Array, points: Points, N: number, _verbose = false, { c = 0 } = {}) => run(scalars, points, N, c),
  };
  return { Parallel };
}

// scripts/zprize23/submission-bls377.ts: byte inputs, points converted once and kept on the GPU
const BLS12_377 = create(Curve.BLS12_377_G1);
let cachedBytes: Uint8Array | undefined, cachedPoints: Points | undefined;
export async function compute_msm(inputPoints: Uint8Array, inputScalars: Uint8Array): Promise<{ x: bigint; y: bigint }> {
  if (cachedBytes !== inputPoints) { cachedPoints = BLS12_377.Parallel.pointsFromBytes(inputPoints); cachedBytes = inputPoints; }
  const { result } = await BLS12_377.Parallel.msmUnsafe(inputScalars, cachedPoints!, inputScalars.length / 32);
  return { x: result.x, y: result.y };
}
