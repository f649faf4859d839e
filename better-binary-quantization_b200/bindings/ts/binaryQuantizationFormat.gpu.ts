/**
 * Drop-in replacement for the class `BinaryQuantizationFormat` of leolee9086/Better-Binary-Quantization
 * (src/binaryQuantizationFormat.ts:132-601): same class name, constructor and ALL TEN public members
 *
 *   quantizeVectors :165            quantizeQueryVector :271          searchNearestNeighbors :308
 *   computeQuantizationAccuracy :420 serializeVectorData :483          deserializeVectorData :533
 *   getConfig :583                  getQuantizer :591                 getScorer :599          (+ the constructor :141)
 *
 * with the same argument meaning, return shapes and error messages.  The class EXTENDS the reference's own class, so
 * every member exists with the reference's exact type (src/index.ts:133 calls computeQuantizationAccuracy; :591 / :599
 * hand out the reference's OptimizedScalarQuantizer / BinaryQuantizedScorer helper objects, which stay what they
 * are); the members ON THE PATH are overridden to run on a B200 through the N-API addon (bindings/napi) and
 * libbbq_b200.so.  There is no JS/WASM fallback behind an overridden member: a failure of the device path throws.
 *
 * Install (INTEGRATION.md): rename the reference's src/binaryQuantizationFormat.ts to
 * src/binaryQuantizationFormat.cpu.ts, save this file as src/binaryQuantizationFormat.ts, add errors.ts, and ship
 * bbq_b200.node + libbbq_b200.so next to dist/.  src/index.ts:20-139 stays byte-for-byte unchanged.
 */
import type {
  BinaryQuantizationConfig, BinarizedByteVectorValues, QuantizationResult, VectorDataFormat, MetadataFormat
} from './types';
import { VectorSimilarityFunction } from './types';
import { QUERY_BITS, INDEX_BITS } from './constants';
import type { OptimizedScalarQuantizer } from './optimizedScalarQuantizer';
import { BinaryQuantizationFormat as ReferenceBinaryQuantizationFormat } from './binaryQuantizationFormat.cpu';
import { toReferenceError } from './errors';

type Handle = unknown;
// eslint-disable-next-line @typescript-eslint/no-var-requires
const addon = require('./bbq_b200.node') as {
  create(queryBits: number, indexBits: number, sim: number, lambda: number, iters: number, device: number): Handle;
  build(ctx: Handle, rows: Float32Array, n: number, dim: number, centroid: Float32Array | null): Handle;
  buildSharded(ctx: Handle, rows: Float32Array, n: number, dim: number, centroid: Float32Array | null): Handle;
  info(index: Handle): { size: number; dimension: number; centroid: Float32Array; centroidDP: number };
  search(index: Handle, queries: Float32Array, nq: number, k: number):
    { indices: Int32Array; scores: Float32Array; count: number; stride: number };
  searchSharded(index: Handle, queries: Float32Array, nq: number, k: number):
    { indices: Int32Array; scores: Float32Array; count: number; stride: number };
  rows(index: Handle, first: number, count: number): { packed: Uint8Array; corrections: Float64Array };
  attachRows(index: Handle, rows: Float32Array): void;
  searchRerank(index: Handle, queries: Float32Array, nq: number, k: number, factor: number):
    { indices: Int32Array; quantizedScores: Float32Array; trueScores: Float64Array; count: number };
  searchRerankSharded(index: Handle, queries: Float32Array, nq: number, k: number, factor: number):
    { indices: Int32Array; quantizedScores: Float32Array; trueScores: Float64Array; count: number };
  saveIndex(index: Handle, veb: string, vemb: string): void;
  loadIndex(ctx: Handle, veb: string, vemb: string): Handle;
  saveIndexSharded(index: Handle, veb: string, vemb: string): void;
  loadIndexSharded(ctx: Handle, veb: string, vemb: string): Handle;
  quantizeQuery(ctx: Handle, query: Float32Array, centroid: Float32Array): { codes: Uint8Array; corrections: Float64Array };
  accuracy(ctx: Handle, rows: Float32Array, queries: Float32Array, n: number, dim: number, targetOrd: number): Float64Array;
  fromQuantized(ctx: Handle, packed: Uint8Array, corrections: Float64Array, centroid: Float32Array, n: number, dim: number): Handle;
  commUniqueId(): Uint8Array;
  commInit(ctx: Handle, id: Uint8Array, rank: number, world: number): void;
  setBase(index: Handle, base: number): void;
  groupCreate(queryBits: number, indexBits: number, sim: number, lambda: number, iters: number, devices: Int32Array): Handle;
  groupContext(group: Handle): Handle;
  groupBuild(group: Handle, rows: Float32Array, n: number, dim: number, centroid: Float32Array | null): Handle;
  groupFromQuantized(group: Handle, packed: Uint8Array, corrections: Float64Array, centroid: Float32Array, n: number, dim: number): Handle;
  groupLoadIndex(group: Handle, veb: string, vemb: string): Handle;
  groupSaveIndex(index: Handle, veb: string, vemb: string): void;
  groupInfo(index: Handle): { size: number; dimension: number; centroid: Float32Array; centroidDP: number };
  groupRows(index: Handle, first: number, count: number): { packed: Uint8Array; corrections: Float64Array };
  groupAttachRows(index: Handle, rows: Float32Array): void;
  groupSearch(index: Handle, queries: Float32Array, nq: number, k: number):
    { indices: Int32Array; scores: Float32Array; count: number; stride: number };
  groupSearchRerank(index: Handle, queries: Float32Array, nq: number, k: number, factor: number):
    { indices: Int32Array; quantizedScores: Float32Array; trueScores: Float64Array; count: number };
};

const SIM_CODE: Record<string, number> = { EUCLIDEAN: 0, COSINE: 1, MAXIMUM_INNER_PRODUCT: 2 };

/** Float32Array[] -> one flat Float32Array, raising the reference's messages (:185-193). */
function flatten(vectors: Float32Array[], dim: number): Float32Array {
  const flat = new Float32Array(vectors.length * dim);
  for (let i = 0; i < vectors.length; i++) {
    const v = vectors[i];
    if (!v) throw new Error(`向量 ${i} 不能为空`);
    if (v.length !== dim) throw new Error(`向量 ${i} 维度 ${v.length} 与第一个向量维度 ${dim} 不匹配`);
    flat.set(v, i * dim);
  }
  return flat;
}

/** src/binaryQuantizationFormat.ts:24-126 — the index now lives in HBM; this object is a handle.  `grouped`: an index
 *  of a device group, one row shard per GPU (its members read through the group entries). */
class DeviceBinarizedByteVectorValues implements BinarizedByteVectorValues {
  private readonly meta: { size: number; dimension: number; centroid: Float32Array; centroidDP: number };
  constructor(public readonly handle: Handle, public readonly grouped = false) {
    this.meta = grouped ? addon.groupInfo(handle) : addon.info(handle);
  }
  rows(first: number, count: number): { packed: Uint8Array; corrections: Float64Array } {
    return this.grouped ? addon.groupRows(this.handle, first, count) : addon.rows(this.handle, first, count);
  }
  dimension(): number { return this.meta.dimension; }                       // :45
  size(): number { return this.meta.size; }                                 // :49
  getCentroid(): Float32Array { return this.meta.centroid; }                // :123
  getCentroidDP(queryVector?: Float32Array): number {                       // :113-121
    if (!queryVector) return this.meta.centroidDP;
    let s = 0;
    for (let i = 0; i < queryVector.length; i++) s += queryVector[i]! * this.meta.centroid[i]!;
    return s;
  }
  vectorValue(ord: number): Uint8Array {                                    // :53 (lazy device->host copy)
    if (ord < 0 || ord >= this.meta.size) throw new Error(`向量索引 ${ord} 不存在`);
    return this.rows(ord, 1).packed;
  }
  getUnpackedVector(ord: number): Uint8Array {                              // :68
    if (ord < 0 || ord >= this.meta.size) throw new Error(`未打包向量索引 ${ord} 不存在`);
    const packed = this.vectorValue(ord);
    const out = new Uint8Array(this.meta.dimension);
    for (let i = 0; i < out.length; i++) out[i] = (packed[i >> 3]! >> (7 - (i & 7))) & 1;
    return out;
  }
  getCorrectiveTerms(ord: number): QuantizationResult {                     // :105
    if (ord < 0 || ord >= this.meta.size) throw new Error(`修正项索引 ${ord} 不存在`);
    const c = this.rows(ord, 1).corrections;
    return { lowerInterval: c[0]!, upperInterval: c[1]!, additionalCorrection: c[2]!, quantizedComponentSum: c[3]! };
  }
  clearUnpackedVectorCache(): void { /* nothing is cached on the host */ }
}

function deviceIndex(targetVectors: BinarizedByteVectorValues): DeviceBinarizedByteVectorValues {
  if (!(targetVectors instanceof DeviceBinarizedByteVectorValues))
    throw new Error('[bbq-b200] 目标向量集合 is not a device index (build it with quantizeVectors / deserializeVectorData of this class)');
  return targetVectors;
}
function deviceHandle(targetVectors: BinarizedByteVectorValues): Handle { return deviceIndex(targetVectors).handle; }

/** The GPUs of a device group: config.devices, else BBQ_DEVICES=0,1,... in the environment; null without either. */
function groupDevices(config: BinaryQuantizationConfig): number[] | null {
  const given = (config as BinaryQuantizationConfig & { devices?: number[] }).devices;
  if (given !== undefined && given !== null) return given;
  const env = process.env.BBQ_DEVICES;
  if (env === undefined || env.trim() === '') return null;
  return env.split(',').map((d) => Number(d.trim()));
}
const GROUP_NOT_SHARDED = '[bbq-b200] this format drives a device group, which is already sharded over its GPUs: ' +
  'sharded = true and joinShardGroup do not apply';

export class BinaryQuantizationFormat extends ReferenceBinaryQuantizationFormat {
  private readonly ctx: Handle;
  /** A device group over config.devices / BBQ_DEVICES (one process, every GPU listed), or null: one GPU. */
  private readonly group: Handle | null = null;

  constructor(config: BinaryQuantizationConfig) {                            // :141-158 (super validates 1..8)
    super(config);
    const cfg = { queryBits: QUERY_BITS, indexBits: INDEX_BITS, ...config };
    const q = config.quantizer;
    const sim = SIM_CODE[q.similarityFunction ?? VectorSimilarityFunction.EUCLIDEAN]!;
    const devices = groupDevices(config);
    try {
      if (devices === null) {
        this.ctx = addon.create(cfg.queryBits!, cfg.indexBits!, sim, q.lambda ?? 0.1, q.iters ?? 5,
          Number(process.env.BBQ_DEVICE ?? -1));
      } else {
        this.group = addon.groupCreate(cfg.queryBits!, cfg.indexBits!, sim, q.lambda ?? 0.1, q.iters ?? 5,
          Int32Array.from(devices));
        this.ctx = addon.groupContext(this.group);   // the group's first GPU: quantizeQueryVector, accuracy
      }
    } catch (e) { throw toReferenceError(e, 'build'); }
  }

  /** With sharded = true (after joinShardGroup) the build is collective: every rank passes its own rows, ranks hold
   *  consecutive row ranges in rank order, and a rank may pass none.  Every rank gets the centroid of the whole corpus
   *  and its rows of the whole-corpus index, its base row set. */
  public override quantizeVectors(vectors: Float32Array[], sharded = false): {              // :165-263
    quantizedVectors: BinarizedByteVectorValues; queryQuantizer: OptimizedScalarQuantizer;
  } {
    if (this.group !== null && sharded) throw new Error(GROUP_NOT_SHARDED);
    if (vectors.length === 0 && !sharded) throw new Error('向量集合不能为空');
    const dim = vectors.length === 0 ? 0 : vectors[0]!.length;
    const flat = flatten(vectors, dim);
    try {
      if (this.group !== null) {
        const handle = addon.groupBuild(this.group, flat, vectors.length, dim, null);
        return { quantizedVectors: new DeviceBinarizedByteVectorValues(handle, true), queryQuantizer: this.getQuantizer() };
      }
      const handle = sharded ? addon.buildSharded(this.ctx, flat, vectors.length, dim, null)
                             : addon.build(this.ctx, flat, vectors.length, dim, null);
      // :261 hands out `this.quantizer` (an OptimizedScalarQuantizer): the inherited helper object, as getQuantizer() does
      return { quantizedVectors: new DeviceBinarizedByteVectorValues(handle), queryQuantizer: this.getQuantizer() };
    } catch (e) { throw toReferenceError(e, 'build'); }
  }

  public override quantizeQueryVector(queryVector: Float32Array, centroid: Float32Array): {   // :271-299
    quantizedQuery: Uint8Array; queryCorrections: QuantizationResult;
  } {
    try {
      const r = addon.quantizeQuery(this.ctx, queryVector, centroid);
      const c = r.corrections;
      return { quantizedQuery: r.codes, queryCorrections: {
        lowerInterval: c[0]!, upperInterval: c[1]!, additionalCorrection: c[2]!, quantizedComponentSum: c[3]! } };
    } catch (e) { throw toReferenceError(e, 'search'); }
  }

  public override searchNearestNeighbors(queryVector: Float32Array, targetVectors: BinarizedByteVectorValues, k: number):
      Array<{ index: number; score: number; originalScore?: number }> {      // :308-412
    if (!queryVector) throw new Error('查询向量不能为空');
    if (!targetVectors) throw new Error('目标向量集合不能为空');
    if (k < 0) throw new Error('k值不能为负数');
    if (queryVector.length !== targetVectors.dimension()) throw new Error('查询向量维度与目标向量维度不匹配');
    if (k === 0) return [];
    try {
      // a fractional k: the reference's heap loop (`size() < k2`, :386-389) ends up with ceil(k) results
      const ix = deviceIndex(targetVectors);
      const r = ix.grouped ? addon.groupSearch(ix.handle, queryVector, 1, Math.ceil(k))
                           : addon.search(ix.handle, queryVector, 1, Math.ceil(k));
      const out = new Array(r.count);
      for (let i = 0; i < r.count; i++) out[i] = { index: r.indices[i]!, score: r.scores[i]! };
      return out;
    } catch (e) { throw toReferenceError(e, 'search'); }
  }

  public override computeQuantizationAccuracy(originalVectors: Float32Array[], queryVectors: Float32Array[]): {  // :420-475
    meanError: number; maxError: number; minError: number; stdError: number; correlation: number;
  } {
    if (originalVectors.length === 0) throw new Error('原始向量集合不能为空');
    if (queryVectors.length === 0) throw new Error('查询向量集合不能为空');
    if (originalVectors.length !== queryVectors.length) throw new Error('原始向量集合和查询向量集合长度不匹配');
    const bits = this.getConfig().queryBits ?? QUERY_BITS;
    if (bits !== 1 && bits !== 4) throw new Error(`不支持的查询位数: ${bits}，只支持1位和4位`);   // binaryQuantizedScorer.ts:96
    const dim = originalVectors[0]!.length;
    try {
      const s = addon.accuracy(this.ctx, flatten(originalVectors, dim), flatten(queryVectors, dim),
        originalVectors.length, dim, 0);
      return { meanError: s[0]!, maxError: s[1]!, minError: s[2]!, stdError: s[3]!, correlation: s[4]! };
    } catch (e) { throw toReferenceError(e, 'build'); }
  }

  public override serializeVectorData(vectors: Float32Array[]): { vectorData: VectorDataFormat[]; metadata: MetadataFormat } {  // :483-525
    const { quantizedVectors } = this.quantizeVectors(vectors);
    const n = quantizedVectors.size(), centroid = quantizedVectors.getCentroid();
    const all = deviceIndex(quantizedVectors).rows(0, n);
    const p = Math.ceil(centroid.length / 8);
    const vectorData: VectorDataFormat[] = [];
    for (let i = 0; i < n; i++) {
      vectorData.push({
        binaryValues: all.packed.slice(i * p, (i + 1) * p),   // the packed MSB-first row (the reference re-packs it: a no-use quirk)
        lowerInterval: all.corrections[4 * i]!, upperInterval: all.corrections[4 * i + 1]!,
        additionalCorrection: all.corrections[4 * i + 2]!, quantizedComponentSum: all.corrections[4 * i + 3]! });
    }
    const metadata: MetadataFormat = {
      fieldNumber: 0, vectorEncodingOrdinal: 0, vectorSimilarityOrdinal: 0, dimensions: centroid.length,
      vectorDataOffset: 0, vectorDataLength: 0, vectorCount: n, centroid,
      centroidSquareMagnitude: quantizedVectors.getCentroidDP() };
    return { vectorData, metadata };
  }

  public override deserializeVectorData(vectorData: VectorDataFormat[], metadata: MetadataFormat): BinarizedByteVectorValues {  // :533-560
    const n = vectorData.length, dim = metadata.dimensions, p = Math.ceil(dim / 8);
    const packed = new Uint8Array(n * p), corr = new Float64Array(n * 4);
    vectorData.forEach((d, i) => {
      packed.set(d.binaryValues.subarray(0, p), i * p);
      corr.set([d.lowerInterval, d.upperInterval, d.additionalCorrection, d.quantizedComponentSum], 4 * i);
    });
    try {
      if (this.group !== null)
        return new DeviceBinarizedByteVectorValues(addon.groupFromQuantized(this.group, packed, corr, metadata.centroid, n, dim), true);
      return new DeviceBinarizedByteVectorValues(addon.fromQuantized(this.ctx, packed, corr, metadata.centroid, n, dim));
    } catch (e) { throw toReferenceError(e, 'build'); }
  }

  // getConfig :583, getQuantizer :591, getScorer :599 are inherited unchanged.

  // ---- additive members (not in the reference) --------------------------------------------------------------

  /** A batch of queries in one call; row i equals searchNearestNeighbors(queries[i], ...). */
  public searchBatch(queries: Float32Array[], targetVectors: BinarizedByteVectorValues, k: number, sharded = false) {
    if (this.group !== null && sharded) throw new Error(GROUP_NOT_SHARDED);
    const dim = targetVectors.dimension();
    const flat = new Float32Array(queries.length * dim);
    queries.forEach((q, i) => {
      if (q.length !== dim) throw new Error('查询向量维度与目标向量维度不匹配');
      flat.set(q, i * dim);
    });
    try {
      const ix = deviceIndex(targetVectors), h = ix.handle;
      const r = ix.grouped ? addon.groupSearch(h, flat, queries.length, k)
              : sharded ? addon.searchSharded(h, flat, queries.length, k) : addon.search(h, flat, queries.length, k);
      return queries.map((_, i) => Array.from({ length: r.count }, (_u, j) =>
        ({ index: r.indices[i * r.stride + j]!, score: r.scores[i * r.stride + j]! })));
    } catch (e) { throw toReferenceError(e, 'search'); }
  }

  /** Sharded search over the GPUs of one box (one Node process per GPU; SURVEY §8e).  Rank 0 creates the id and
   *  ships it to its peers (IPC message / env var / file); every rank then joins and declares its shard's base row.
   *  After that searchBatch(..., sharded = true) returns, on every rank, the lists of the whole corpus.  A rank that is
   *  about to load its shard with loadIndex(prefix, true) has no shard yet: it joins without one (the load sets the
   *  base). */
  public static createShardGroupId(): Uint8Array { return addon.commUniqueId(); }
  public joinShardGroup(id: Uint8Array, rank: number, world: number, shard?: BinarizedByteVectorValues, baseRow?: number): void {
    if (this.group !== null) throw new Error(GROUP_NOT_SHARDED);
    try {
      addon.commInit(this.ctx, id, rank, world);
      if (shard !== undefined) addon.setBase(deviceHandle(shard), baseRow ?? 0);
    } catch (e) { throw toReferenceError(e, 'build'); }
  }

  /** getOversampledTopKWithSort / ...WithHeap (src/topKSelector.ts:29-114) on the device: quantised top k*factor,
   *  exact cosine against the attached original rows, best k by true score. */
  public attachOriginalVectors(targetVectors: BinarizedByteVectorValues, vectors: Float32Array[]): void {
    const flat = flatten(vectors, targetVectors.dimension());
    try {
      const ix = deviceIndex(targetVectors);
      if (ix.grouped) addon.groupAttachRows(ix.handle, flat);
      else addon.attachRows(ix.handle, flat);
    }
    catch (e) { throw toReferenceError(e, 'build'); }
  }
  /** With sharded = true (after joinShardGroup, each rank's own rows attached) the re-rank runs over ALL row shards
   *  of the box and returns, on every rank, what the unsharded call returns on the whole corpus. */
  public searchOversampled(queryVector: Float32Array, targetVectors: BinarizedByteVectorValues, k: number,
      oversampleFactor: number, sharded = false): Array<{ index: number; quantizedScore: number; trueScore: number }> {
    if (this.group !== null && sharded) throw new Error(GROUP_NOT_SHARDED);
    try {
      const ix = deviceIndex(targetVectors), h = ix.handle;
      const r = ix.grouped ? addon.groupSearchRerank(h, queryVector, 1, k, oversampleFactor)
              : sharded ? addon.searchRerankSharded(h, queryVector, 1, k, oversampleFactor)
                        : addon.searchRerank(h, queryVector, 1, k, oversampleFactor);
      return Array.from({ length: r.count }, (_u, i) =>
        ({ index: r.indices[i]!, quantizedScore: r.quantizedScores[i]!, trueScore: r.trueScores[i]! }));
    } catch (e) { throw toReferenceError(e, 'search'); }
  }

  /** On-disk form of serializeVectorData / deserializeVectorData (:483-560): `${prefix}.veb` + `${prefix}.vemb`
   *  (FILE_EXTENSIONS, src/constants.ts:52-57), streamed between the files and device memory natively.
   *  With sharded = true (after joinShardGroup) both are collective: every rank saves its own rows into ONE image of
   *  the whole corpus, or loads its own row range of one image (its base set), on any number of ranks. */
  public saveIndex(targetVectors: BinarizedByteVectorValues, prefix: string, sharded = false): void {
    if (this.group !== null && sharded) throw new Error(GROUP_NOT_SHARDED);
    try {
      const ix = deviceIndex(targetVectors), h = ix.handle;
      if (ix.grouped) addon.groupSaveIndex(h, `${prefix}.veb`, `${prefix}.vemb`);
      else if (sharded) addon.saveIndexSharded(h, `${prefix}.veb`, `${prefix}.vemb`);
      else addon.saveIndex(h, `${prefix}.veb`, `${prefix}.vemb`);
    } catch (e) { throw toReferenceError(e, 'build'); }
  }
  public loadIndex(prefix: string, sharded = false): BinarizedByteVectorValues {
    if (this.group !== null && sharded) throw new Error(GROUP_NOT_SHARDED);
    try {
      if (this.group !== null)
        return new DeviceBinarizedByteVectorValues(addon.groupLoadIndex(this.group, `${prefix}.veb`, `${prefix}.vemb`), true);
      const h = sharded ? addon.loadIndexSharded(this.ctx, `${prefix}.veb`, `${prefix}.vemb`)
                        : addon.loadIndex(this.ctx, `${prefix}.veb`, `${prefix}.vemb`);
      return new DeviceBinarizedByteVectorValues(h);
    } catch (e) { throw toReferenceError(e, 'build'); }
  }
}
