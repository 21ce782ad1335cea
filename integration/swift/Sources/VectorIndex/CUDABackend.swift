// CUDABackend.swift -- the reference-side shim a maintainer would add next to
// Sources/VectorIndex/Operations/Quantization/PQEncode+CBackend.swift (same run-time gate pattern, :16-23).
// NOT compiled in this repository (no Swift toolchain in the image); every C entry point used here is exercised through
// the same C ABI by tests/ (ctypes) and by tests/c/abi_smoke.c (plain C).
#if canImport(CVIndexCUDA)
import CVIndexCUDA
#endif

@usableFromInline internal var _useCUDA: Bool {
    #if canImport(CVIndexCUDA)
    return !_envFlag("VECTORINDEX_DISABLE_CUDA") && vix_device_count() > 0
    #else
    return false
    #endif
}

#if canImport(CVIndexCUDA)
@inline(__always) internal func _vixCheck(_ status: Int32, _ what: StaticString) throws {
    guard status >= 0 else {                       // negative = KMeansMBStatus extended (include/vindex_cuda.h)
        throw ErrorBuilder(.internalError, operation: "\(what)")
            .message(String(cString: vix_last_error())).build()
    }
}

// ivf_select_nprobe_batch_f32 (Kernels/IVFSelect.swift:242-253)
public func ivf_select_nprobe_batch_f32_cuda(Q: UnsafePointer<Float>, b: Int, d: Int,
                                             centroids: UnsafePointer<Float>, kc: Int, metric: IVFMetric, nprobe: Int,
                                             centroidNorms: UnsafePointer<Float>?, disabledLists: UnsafePointer<UInt64>?,
                                             listIDsOut: UnsafeMutablePointer<Int32>,
                                             listScoresOut: UnsafeMutablePointer<Float>?) throws {
    try _vixCheck(vix_ivf_select_nprobe_batch_f32(Q, Int64(b), Int32(d), centroids, Int32(kc),
                                                  metric == .l2 ? 0 : 1, Int32(nprobe), centroidNorms, disabledLists,
                                                  listIDsOut, listScoresOut), "ivf_select_nprobe_batch_f32")
    // The library orders and reports in the batchSearch convention ("smaller is better": ||c||^2 - 2<q,c>, -<q,c>;
    // CentroidBatchScore.swift:54-64).  The lists are IVFSelect's (same order, same tie rule); its listScoresOut are
    // ||q||^2 + ||c||^2 - 2<q,c> and <q,c> (IVFSelect.swift:436-479): restore them here.
    guard let scores = listScoresOut else { return }
    for qi in 0..<b {
        let qn: Float = metric == .l2 ? IndexOps.Support.Norms.l2NormSquared(vector: Q + qi * d, dimension: d) : 0
        for p in 0..<nprobe where listIDsOut[qi * nprobe + p] >= 0 {
            scores[qi * nprobe + p] = metric == .l2 ? qn + scores[qi * nprobe + p] : -scores[qi * nprobe + p]
        }
    }
}

// adc_scan_u8 (Operations/Quantization/ADCScan.swift:99-121)
public func adc_scan_u8_cuda(codes: UnsafePointer<UInt8>, n: Int, m: Int, ks: Int, lut: UnsafePointer<Float>,
                             out: UnsafeMutablePointer<Float>, opts: ADCScanOpts) throws {
    var o = vix_adc_scan_opts()
    o.layout = Int32(opts.layout.rawValue); o.group_size = Int32(opts.groupSize); o.stride = Int32(opts.stride)
    o.add_bias = opts.addBias; o.strict_fp = opts.strictFP          // ADCScanOpts (ADCScan.swift:23-49); addBias is a Float
    try _vixCheck(vix_adc_scan_u8(codes, Int64(n), Int32(m), Int32(ks), lut, out, &o), "adc_scan_u8")
}

/// Whole-query offload: the device-resident counterpart of the IVFIndex actor's lists (IVFIndex.swift:42).
public final class CUDAIVFPQIndex {
    private var h: OpaquePointer?

    public init(dimension: Int, metric: SupportedDistanceMetric, nlist: Int, nprobe: Int, m: Int) throws {
        var p = vix_index_params(); vix_index_params_default(&p)
        p.kind = 2; p.d = Int32(dimension); p.metric = metric == .euclidean ? 0 : 1
        p.nlist = Int32(nlist); p.nprobe = Int32(nprobe); p.m = Int32(m)
        try _vixCheck(vix_index_create(&p, &h), "vix_index_create")
    }
    deinit { vix_index_destroy(h) }

    public func optimize(_ x: [Float], count: Int) throws {
        try _vixCheck(vix_index_train(h, x, Int64(count), nil, nil), "vix_index_train")
    }
    public func batchInsert(_ x: [Float], ids: [Int64]) throws {
        try _vixCheck(vix_index_add(h, x, ids, Int64(ids.count)), "vix_index_add")
    }
    /// remove(id:) for a batch: every stored row whose id is listed goes; returns the number of rows removed
    public func batchRemove(ids: [Int64]) throws -> Int {
        var removed: Int64 = 0
        try _vixCheck(vix_index_remove(h, ids, Int64(ids.count), &removed), "vix_index_remove")
        return Int(removed)
    }
    /// ascending by API distance, padded with id -1 / NaN; k <= 0 leaves the outputs untouched (IVFIndex.swift:866)
    public func batchSearch(_ q: [Float], nq: Int, k: Int) throws -> ([Float], [Int64]) {
        var dist = [Float](repeating: .nan, count: nq * k); var ids = [Int64](repeating: -1, count: nq * k)
        try _vixCheck(vix_index_search(h, q, Int64(nq), Int32(k), 0, &dist, &ids), "vix_index_search")
        return (dist, ids)
    }
    /// `filter:` closures become an IDFilterBitset over the actor's dense ids (Operations/Filtering/IDFilter.swift)
    public func batchSearch(_ q: [Float], nq: Int, k: Int, allow: IDFilterBitset) throws -> ([Float], [Int64]) {
        var dist = [Float](repeating: .nan, count: nq * k); var ids = [Int64](repeating: -1, count: nq * k)
        try _vixCheck(vix_index_search_filtered(h, q, Int64(nq), Int32(k), 0, allow.readOnly, Int64(allow.capacity),
                                                Int32(VIX_FILTER_ALLOW.rawValue), &dist, &ids), "vix_index_search_filtered")
        return (dist, ids)
    }
    // step 7 of the IVF-PQ query (docs/kernel-specs/DONE_22_adc_scan.md:873-878): ADC top-R, then Kernel #40 over the
    // original vectors (DenseArray reader: id = row of `vectors`); raw exact scores out (L2^2 / dot), best first
    public func batchSearchReranked(_ q: [Float], nq: Int, k: Int, rerankR: Int, vectors: UnsafePointer<Float>, count: Int)
        throws -> ([Float], [Int64]) {
        var sc = [Float](repeating: .infinity, count: nq * k); var ids = [Int64](repeating: -1, count: nq * k)
        try _vixCheck(vix_index_search_rerank(h, q, Int64(nq), Int32(k), 0, Int32(rerankR), vectors, Int64(count), nil, &sc, &ids),
                      "search_rerank")
        return (sc, ids)
    }

    // ---- one process per GPU: the inverted lists sharded over the ranks of a vix_comm_t (csrc/vix_sharded.cu) ----
    // `id`: the 128 bytes rank 0 obtained from vix_comm_unique_id and handed to every worker by the host's own means
    public static func makeComm(id: [UInt8], rank: Int, world: Int) throws -> OpaquePointer? {
        var c: OpaquePointer?
        try _vixCheck(vix_comm_create(id, id.count, Int32(rank), Int32(world), &c), "comm_create")
        return c
    }
    public func shardedInsert(_ comm: OpaquePointer?, _ x: [Float], ids: [Int64]) throws {      // collective
        try _vixCheck(vix_sharded_add(h, comm, nil, x, ids, Int64(ids.count)), "sharded_add")
    }
    public func shardedSearch(_ comm: OpaquePointer?, _ q: [Float], nq: Int, k: Int) throws -> ([Float], [Int64]) {   // collective
        var dist = [Float](repeating: .nan, count: nq * k); var ids = [Int64](repeating: -1, count: nq * k)
        try _vixCheck(vix_sharded_search(h, comm, q, Int64(nq), Int32(k), 0, &dist, &ids), "sharded_search")
        return (dist, ids)
    }
}
#endif
