// fsharp/GibbsSamplingB200.fs -- the reference-side binding (NOT compiled in this repository: the
// image has no .NET toolchain; the Python twin of this file is gibbssampling_b200/SiteSampler.py).
//
// Drop-in for the SiteSampler and MotifSampler modules of GibbsSampling.fs: same module names, function names, argument
// order and result types; the body of each function marshals its arguments to libgibbs_b200.so
// (include/gibbs_b200.h, ABI version 2) with P/Invoke instead of running the F# loops. `seed` is the one addition:
// the reference builds `System.Random()` from the clock (fs:144, fs:829), which cannot be reproduced.
// The restart loops (numberOfRepetitions) spread their restarts over every GPU of the box (gibbs_multi_*).
namespace GibbsSampling

open System
open System.Runtime.InteropServices
open BioFSharp

module Native =

    [<Struct; StructLayout(LayoutKind.Sequential)>]
    type GibbsParams =
        val mutable k             : int
        val mutable alphabetSize  : int
        val mutable pseudocount   : float
        val mutable bgA           : float
        val mutable bgC           : float
        val mutable bgG           : float
        val mutable bgT           : float
        val mutable cutoff        : float
        val mutable sampler       : int
        val mutable phaseShifts   : int
        val mutable maxSweeps     : int
        val mutable phaseMask     : int
        val mutable background    : int   // 0 = fixed pcv (WithBPV), 1 = data-derived (fs:697)
        val mutable motifAmount   : int   // MotifSampler motifAmount: 0 / 1 = one site per sequence, 2 = up to two (fs:727-742)

    [<Struct; StructLayout(LayoutKind.Sequential)>]
    type GibbsRunStats =
        val mutable siteUpdates   : int64
        val mutable windowScores  : int64
        val mutable sweeps        : int64
        val mutable exactRescans  : int64
        val mutable cappedChains  : int64
        val mutable specDiscards  : int64
        val mutable kernelLaunches: int
        val mutable fastPath      : int
        val mutable teamWarps     : int
        val mutable initPath      : int   // GIBBS_INIT_CHAIN / _WIDE / _SMEM / _TILED
        val mutable kernelMs      : float

    [<Literal>]
    let Lib = "gibbs_b200" // libgibbs_b200.so next to GibbsSampling.dll

    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern IntPtr gibbs_last_error()
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_create(byte[] seqs, int64[] offsets, int nSeqs, int device, IntPtr& handle)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_destroy(IntPtr handle)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_set_start_state(IntPtr handle, int nChains, int[] sites, float[] scores)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_set_start_ppm(IntPtr handle, float[] ppmOrNull, int k)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_host_alloc(unativeint bytes, IntPtr& ptr)   // optional: page-locked result buffers
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_host_free(IntPtr ptr)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_fetch(IntPtr handle, int[] sitesOut, float[] scoresOut, float[] sumsOut, int& bestChain, int[] countsOut, GibbsRunStats& stats)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_pick_argmax(IntPtr handle, int[] sites, int heldout, GibbsParams& p, float& score, int& site)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_run(IntPtr handle, GibbsParams& p, int nChains, int64 chainIdBase, uint64 seed, int rngMode,
                         float[] uniformsOrNull, int64 uniformsPerChain, int[] sitesOut, float[] scoresOut,
                         float[] sumsOut, int& bestChain, int[] countsOut, GibbsRunStats& stats)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_set_start_motif_state(IntPtr handle, int nChains, int m, int[] positions, float[] pwms)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_fetch_positions(IntPtr handle, int m, int[] positionsOut)
    // restart loops: one process, every GPU of the box (the restart axis of fsx:430 / fsx:1162); the promote-or-restart
    // loop of fs:435-459 is decided by the library, only its result comes back
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_create(byte[] seqs, int64[] offsets, int nSeqs, int[] devicesOrNull, int nDevices, IntPtr& multi)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_destroy(IntPtr multi)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_num_devices(IntPtr multi)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern IntPtr gibbs_multi_handle(IntPtr multi, int slot)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_run_device(IntPtr multi, GibbsParams& p, int nChains, int64 chainIdBase, uint64 seed, int rngMode,
                                      float[] uniformsOrNull, int64 uniformsPerChain)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_fetch_best(IntPtr multi, int repetitions, int[] sitesOut, float[] scoresOut, int& nOut, float& sumOut,
                                      int& restartOut, int[] countsOut, GibbsRunStats& stats)
    // the same on one handle (motifAmount = 2 returns Positions lists through gibbs_fetch_best_positions)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_run_device(IntPtr handle, GibbsParams& p, int nChains, int64 chainIdBase, uint64 seed, int rngMode,
                                float[] uniformsOrNull, int64 uniformsPerChain)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_fetch_best(IntPtr handle, int repetitions, int[] sitesOut, float[] scoresOut, int& nOut, float& sumOut,
                                int& restartOut, int[] countsOut, GibbsRunStats& stats)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_fetch_best_positions(IntPtr handle, int m, int[] positionsOut)
    // many sequence sets in one batch (include/gibbs_b200.h, gibbs_batch_*)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_create(byte[] seqs, int64[] offsets, int[] setOffsets, int nSets, int device, IntPtr& batch)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_destroy(IntPtr batch)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_run_device(IntPtr batch, GibbsParams& p, float[] bgPerSetOrNull, int restartsPerSet, int64 chainIdBase, uint64 seed)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_fetch(IntPtr batch, int[] sitesOut, float[] scoresOut, float[] sumsOut, GibbsRunStats& stats)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_fetch_best(IntPtr batch, int repetitions, int[] sitesOut, float[] scoresOut, int[] nOut, float[] sumOut,
                                      int[] restartOut, int[] countsOut, GibbsRunStats& stats)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_run_motif_device(IntPtr batch, GibbsParams& p, float[] bgPerSetOrNull, int restartsPerSet, int64 chainIdBase,
                                            uint64 seed)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_fetch_positions(IntPtr batch, int m, int[] positionsOut)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_batch_fetch_best_positions(IntPtr batch, int m, int[] positionsOut)
    // the same batch with its sets split over every GPU of the box (gibbs_multi_batch_*): outputs in the caller's set order
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_create(byte[] seqs, int64[] offsets, int[] setOffsets, int nSets, int[] devicesOrNull, int nDevices,
                                        IntPtr& multiBatch)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_destroy(IntPtr multiBatch)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_num_devices(IntPtr multiBatch)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_slot_sets(IntPtr multiBatch, int slot, int& firstSet, int& nSets)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_run_device(IntPtr multiBatch, GibbsParams& p, float[] bgPerSetOrNull, int restartsPerSet,
                                            int64 chainIdBase, uint64 seed)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_run_motif_device(IntPtr multiBatch, GibbsParams& p, float[] bgPerSetOrNull, int restartsPerSet,
                                                  int64 chainIdBase, uint64 seed)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_fetch(IntPtr multiBatch, int[] sitesOut, float[] scoresOut, float[] sumsOut, GibbsRunStats& stats)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_fetch_best(IntPtr multiBatch, int repetitions, int[] sitesOut, float[] scoresOut, int[] nOut,
                                            float[] sumOut, int[] restartOut, int[] countsOut, GibbsRunStats& stats)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_fetch_positions(IntPtr multiBatch, int m, int[] positionsOut)
    [<DllImport(Lib, CallingConvention = CallingConvention.Cdecl)>]
    extern int gibbs_multi_batch_fetch_best_positions(IntPtr multiBatch, int m, int[] positionsOut)

    /// status code -> the exception the reference would have thrown (SURVEY.md section 8b)
    let check (rc:int) =
        if rc <> 0 then
            let msg = Marshal.PtrToStringAnsi(gibbs_last_error())
            match rc with
            | 1 -> raise (ArgumentException msg)
            | 2 -> raise (IndexOutOfRangeException msg)        // symbol outside the table, fs:17
            | 3 -> raise (InvalidOperationException msg)       // Array.take on a short sequence, fs:152
            | 7 -> raise (ArgumentException msg)               // roulette pick beyond the mass, fs:753
            | 8 -> raise (NotSupportedException msg)
            | _ -> raise (ExternalException(msg, rc))          // CUDA failure; there is no CPU fallback

    /// sources : BioArray<#IBioItem>[] -> one ASCII buffer + offsets (BioItem.symbol, fs:17)
    let flatten (sources:BioArray.BioArray<#IBioItem>[]) =
        let offsets = Array.zeroCreate<int64> (sources.Length + 1)
        sources |> Array.iteri (fun i s -> offsets.[i + 1] <- offsets.[i] + int64 s.Length)
        let buf = Array.zeroCreate<byte> (int offsets.[sources.Length])
        sources |> Array.iteri (fun i s -> s |> Array.iteri (fun j b -> buf.[int offsets.[i] + j] <- byte (BioItem.symbol b)))
        buf, offsets

    /// pcv = Some _ : the WithBPV family (fixed background); None : the data-derived family (fs:462, fs:697)
    let makeParams (k:int) (pc:float) (alphabet:#IBioItem[]) (pcv:CompositeVector.ProbabilityCompositeVector option) phaseMask =
        let mutable p = GibbsParams()
        p.k <- k; p.alphabetSize <- alphabet.Length; p.pseudocount <- pc
        match pcv with
        | Some v ->
            let sym c = v.Array.[int c - 42]
            p.bgA <- sym 'A'; p.bgC <- sym 'C'; p.bgG <- sym 'G'; p.bgT <- sym 'T'; p.background <- 0
        | None ->
            p.bgA <- 0.25; p.bgC <- 0.25; p.bgG <- 0.25; p.bgT <- 0.25; p.background <- 1
        p.sampler <- 0; p.phaseShifts <- 1; p.maxSweeps <- 0; p.phaseMask <- phaseMask
        p

    /// rows A,C,G,T of a 49 x k PositionProbabilityMatrix as [k][4] (gibbs_set_start_ppm)
    let flattenPPM (k:int) (ppM:PositionMatrix.PositionProbabilityMatrix) =
        Array.init (k * 4) (fun e -> ppM.Matrix.[int "ACGT".[e % 4] - 42, e / 4])

    /// n restarts as n chains of one launch; returns (scores, sites, sums) per restart
    let runChainsWith (ppM:PositionMatrix.PositionProbabilityMatrix option) (phaseMask:int) (nChains:int) (seed:uint64) k pc alphabet sources
                      (pcv:CompositeVector.ProbabilityCompositeVector option) (start:((float*int)[]) option) =
        let buf, offsets = flatten sources
        let mutable h = IntPtr.Zero
        check (gibbs_create(buf, offsets, sources.Length, 0, &h))
        try
            let n = sources.Length
            match start with
            | Some st ->
                let sites  = Array.init (nChains * n) (fun i -> snd st.[i % n])
                let scores = Array.init (nChains * n) (fun i -> fst st.[i % n])
                check (gibbs_set_start_state(h, nChains, sites, scores))
            | None -> ()
            match ppM with
            | Some m -> check (gibbs_set_start_ppm(h, flattenPPM k m, k))   // fs:644: positionProbabilityMatrix
            | None -> ()
            let mutable p = makeParams k pc alphabet pcv phaseMask
            let sites, scores, sums = Array.zeroCreate (nChains * n), Array.zeroCreate (nChains * n), Array.zeroCreate nChains
            let mutable best = 0
            let mutable stats = GibbsRunStats()
            check (gibbs_run(h, &p, nChains, 0L, seed, 0, null, 0L, sites, scores, sums, &best, null, &stats))
            Array.init nChains (fun c -> Array.init n (fun i -> scores.[c * n + i], sites.[c * n + i])), sums
        finally
            gibbs_destroy h |> ignore

    let runChains phaseMask nChains seed k pc alphabet sources pcv start =
        runChainsWith None phaseMask nChains seed k pc alphabet sources (Some pcv) start

    /// The restart loops (fs:434, fs:615, fs:664): numberOfRepetitions + 1 restarts over EVERY GPU of the box (one handle per
    /// device, contiguous blocks of restarts, streams keyed by the global restart index); the loop of fs:435-459 is decided
    /// by the library from one sum per restart and only the returned (float*int)[] is copied back.
    let bestOfRestarts (ppM:PositionMatrix.PositionProbabilityMatrix option) (numberOfRepetitions:int) (seed:uint64) k pc alphabet sources
                       (pcv:CompositeVector.ProbabilityCompositeVector option) : (float*int)[] =
        let buf, offsets = flatten sources
        let mutable m = IntPtr.Zero
        check (gibbs_multi_create(buf, offsets, sources.Length, null, 0, &m))   // 0 = every visible device
        try
            let n = sources.Length
            match ppM with
            | Some mat ->
                let flat = flattenPPM k mat
                for slot in 0 .. gibbs_multi_num_devices m - 1 do
                    check (gibbs_set_start_ppm(gibbs_multi_handle(m, slot), flat, k))
            | None -> ()
            let mutable p = makeParams k pc alphabet pcv 0
            check (gibbs_multi_run_device(m, &p, numberOfRepetitions + 1, 0L, seed, 0, null, 0L))
            let sites, scores = Array.zeroCreate n, Array.zeroCreate n
            let mutable nOut = 0
            let mutable sum = 0.
            let mutable restart = 0
            let mutable stats = GibbsRunStats()
            check (gibbs_multi_fetch_best(m, numberOfRepetitions, sites, scores, &nOut, &sum, &restart, null, &stats))
            Array.init nOut (fun i -> scores.[i], sites.[i])     // nOut = 1: the loop's initial value [|(0., 0)|] survived
        finally
            gibbs_multi_destroy m |> ignore

    /// The restart loops of many sets in one batch over EVERY GPU of the box (contiguous blocks of sets, one per device): set s
    /// gets exactly what bestOfRestarts-style single-set calls with the same seed give (restart r of every set draws from the
    /// stream (seed, r)), whatever the number of devices; only the winners are copied back.
    let bestOfRestartsOfSets (numberOfRepetitions:int) (seed:uint64) k pc alphabet (sets:BioArray.BioArray<#IBioItem>[][])
                             (pcvs:CompositeVector.ProbabilityCompositeVector[] option) : (float*int)[][] =
        let all = Array.concat sets
        let buf, offsets = flatten all
        let setOffsets = Array.zeroCreate<int> (sets.Length + 1)
        sets |> Array.iteri (fun s src -> setOffsets.[s + 1] <- setOffsets.[s] + src.Length)
        let mutable b = IntPtr.Zero
        check (gibbs_multi_batch_create(buf, offsets, setOffsets, sets.Length, null, 0, &b))   // 0 = every visible device
        try
            let mutable p = makeParams k pc alphabet (pcvs |> Option.map (fun v -> v.[0])) 0
            let bg =
                match pcvs with
                | Some v -> v |> Array.collect (fun pcv -> [| for c in "ACGT" -> pcv.Array.[int c - 42] |])
                | None -> null
            check (gibbs_multi_batch_run_device(b, &p, bg, numberOfRepetitions + 1, 0L, seed))
            let sites, scores = Array.zeroCreate all.Length, Array.zeroCreate all.Length
            let nOut = Array.zeroCreate sets.Length
            let mutable stats = GibbsRunStats()
            check (gibbs_multi_batch_fetch_best(b, numberOfRepetitions, sites, scores, nOut, null, null, null, &stats))
            Array.init sets.Length (fun s -> Array.init nOut.[s] (fun i -> scores.[setOffsets.[s] + i], sites.[setOffsets.[s] + i]))
        finally
            gibbs_multi_batch_destroy b |> ignore

open CompositeVector

module SiteSampler =

    let private seedOf (seed:uint64 option) = defaultArg seed (uint64 DateTime.Now.Ticks)

    /// fs:412-430
    let getPWMOfRandomStartsWithBPV motifLength pseudoCount alphabet sources (pcv:ProbabilityCompositeVector) =
        (Native.runChains 1 1 (seedOf None) motifLength pseudoCount alphabet sources pcv None |> fst).[0]
    /// fs:381-408
    let findBestMotifWithStartPosition motifLength pseudoCount alphabet sources pcv (startPositions:(float*int)[]) =
        (Native.runChains 2 1 0UL motifLength pseudoCount alphabet sources pcv (Some startPositions) |> fst).[0]
    /// fs:350-377
    let getLeftShiftedBestPWMSsWithBPV motifLength pseudoCount alphabet sources pcv (startPositions:(float*int)[]) =
        (Native.runChains 4 1 0UL motifLength pseudoCount alphabet sources pcv (Some startPositions) |> fst).[0]
    /// fs:318-346
    let getRightShiftedBestPWMSsWithBPV motifLength pseudoCount alphabet sources pcv (startPositions:(float*int)[]) =
        (Native.runChains 8 1 0UL motifLength pseudoCount alphabet sources pcv (Some startPositions) |> fst).[0]
    /// fs:691-695
    let doSiteSamplingWithBPV motifLength pseudoCount alphabet sources (pcv:ProbabilityCompositeVector) =
        (Native.runChains 15 1 (seedOf None) motifLength pseudoCount alphabet sources pcv None |> fst).[0]

    /// fs:434-459. The numberOfRepetitions + 1 restarts the loop can consume run as parallel chains on every GPU of the box;
    /// the loop itself (promote-or-restart, quirk A.6-8) is decided by the library (gibbs_multi_fetch_best).
    let getMotifsWithBestInformationContentWithBPV (numberOfRepetitions:int) motifLength pseudoCount alphabet sources (pcv:ProbabilityCompositeVector) =
        Native.bestOfRestarts None numberOfRepetitions (seedOf None) motifLength pseudoCount alphabet sources (Some pcv)

    /// getMotifsWithBestInformationContentWithBPV of every set (pcvs.[s] the background of sets.[s]) in one batch over every GPU
    let getMotifsWithBestInformationContentWithBPVOfSets (numberOfRepetitions:int) motifLength pseudoCount alphabet sets (pcvs:ProbabilityCompositeVector[]) =
        Native.bestOfRestartsOfSets numberOfRepetitions (seedOf None) motifLength pseudoCount alphabet sets (Some pcvs)

    // ---- data-derived background (fs:462-640, fs:697): background = 1, no pcv ---------------------------------
    // Gap '-' is an alphabet member here when alphabet holds it (dnaBases): gap-padded alignments run with its PWM row.
    /// fs:697-701
    let doSiteSampling motifLength pseudoCount alphabet sources =
        (Native.runChainsWith None 15 1 (seedOf None) motifLength pseudoCount alphabet sources None None |> fst).[0]
    /// fs:703-707 (ppM has no Gap row: sets holding '-' with Gap in the alphabet raise NotSupportedException)
    let doSiteSamplingWithPPM motifLength pseudoCount alphabet sources (ppM:PositionMatrix.PositionProbabilityMatrix) =
        (Native.runChainsWith (Some ppM) 15 1 (seedOf None) motifLength pseudoCount alphabet sources None None |> fst).[0]
    /// fs:644-661 (as doSiteSamplingWithPPM for Gap)
    let getMotifsWithBestPWMSOfPPM motifLength pseudoCount alphabet sources (ppM:PositionMatrix.PositionProbabilityMatrix) =
        (Native.runChainsWith (Some ppM) 1 1 (seedOf None) motifLength pseudoCount alphabet sources None None |> fst).[0]
    /// fs:615-640 -- the script's live call (fsx:384)
    let getMotifsWithBestInformationContent (numberOfRepetitions:int) motifLength pseudoCount alphabet sources =
        Native.bestOfRestarts None numberOfRepetitions (seedOf None) motifLength pseudoCount alphabet sources None
    /// getMotifsWithBestInformationContent of every set in one batch over every GPU
    let getMotifsWithBestInformationContentOfSets (numberOfRepetitions:int) motifLength pseudoCount alphabet sets =
        Native.bestOfRestartsOfSets numberOfRepetitions (seedOf None) motifLength pseudoCount alphabet sets None
    /// fs:664-689
    let getBestInformationContentOfPPM (numberOfRepetitions:int) motifLength pseudoCount alphabet sources (ppM:PositionMatrix.PositionProbabilityMatrix) =
        Native.bestOfRestarts (Some ppM) numberOfRepetitions (seedOf None) motifLength pseudoCount alphabet sources None

module MotifSampler =

    /// fs:712-716 (kept as in the reference)
    type MotifIndex = { PWMS : float; Positions : int list }
    let createMotifIndex pwms pos = { PWMS = pwms; Positions = pos }

    let private seedOf (seed:uint64 option) = defaultArg seed (uint64 DateTime.Now.Ticks)

    /// sampler = 1 (include/gibbs_b200.h); motifAmount 1 or 2 (Positions lists newest first, fs:736; three and more sites per
    /// sequence are GIBBS_ERR_UNSUPPORTED). bestOf = Some numberOfRepetitions: the restart loop (fs:857-881) over nChains
    /// restarts, decided by the library; None: the state of every chain.
    let private run (phaseMask:int) (nChains:int) seed (motifAmount:int) k pc (cutOff:float) alphabet sources
                    (pcv:ProbabilityCompositeVector option) (ppM:PositionMatrix.PositionProbabilityMatrix option) (start:MotifIndex[] option)
                    (bestOf:int option) : MotifIndex[][] =
        let m = max motifAmount 1
        let buf, offsets = Native.flatten sources
        let mutable h = IntPtr.Zero
        Native.check (Native.gibbs_create(buf, offsets, sources.Length, 0, &h))
        try
            let n = sources.Length
            match start with
            | Some st ->   // Positions lists, newest first; -1 = absent (fs:796: a sequence may have no site)
                let pos = Array.init (nChains * n * m) (fun e ->
                              let ps = st.[(e / m) % n].Positions
                              if e % m < ps.Length then ps.[e % m] else -1)
                let pwms = Array.init (nChains * n) (fun i -> st.[i % n].PWMS)
                Native.check (Native.gibbs_set_start_motif_state(h, nChains, m, pos, pwms))
            | None -> ()
            match ppM with
            | Some mat -> Native.check (Native.gibbs_set_start_ppm(h, Native.flattenPPM k mat, k))
            | None -> ()
            let mutable p = Native.makeParams k pc alphabet pcv phaseMask
            p.sampler <- 1; p.cutoff <- cutOff; p.motifAmount <- m
            Native.check (Native.gibbs_run_device(h, &p, nChains, 0L, seed, 0, null, 0L))
            let toIndex (scores:float[]) (pos:int[]) (c:int) =
                Array.init n (fun i -> createMotifIndex scores.[c * n + i] ([ for s in 0 .. m - 1 do
                                                                                let q = pos.[(c * n + i) * m + s]
                                                                                if q >= 0 then yield q ]))
            let mutable stats = Native.GibbsRunStats()
            match bestOf with
            | Some reps ->
                let sites, scores, pos = Array.zeroCreate n, Array.zeroCreate n, Array.zeroCreate (n * m)
                let mutable nOut = 0
                let mutable sum = 0.
                let mutable restart = 0
                Native.check (Native.gibbs_fetch_best(h, reps, sites, scores, &nOut, &sum, &restart, null, &stats))
                if restart < 0 then [| [| createMotifIndex 0. [] |] |]       // loop 0 [||] [|createMotifIndex 0. []|] returned its start
                else
                    Native.check (Native.gibbs_fetch_best_positions(h, m, pos))
                    [| toIndex scores pos 0 |]
            | None ->
                let sites, scores, sums = Array.zeroCreate (nChains * n), Array.zeroCreate (nChains * n), Array.zeroCreate nChains
                let pos = Array.zeroCreate (nChains * n * m)
                let mutable best = 0
                Native.check (Native.gibbs_fetch(h, sites, scores, sums, &best, null, &stats))
                Native.check (Native.gibbs_fetch_positions(h, m, pos))
                Array.init nChains (toIndex scores pos)
        finally
            Native.gibbs_destroy h |> ignore

    /// fs:828-853: the synchronous roulette sweep (GIBBS_PHASE_STOCHASTIC = 16)
    let findBestMotifPositionsWithStartPositionsByPCV motifAmount motifLength pseudoCount cutOff alphabet sources (pcv:ProbabilityCompositeVector) (motifMem:MotifIndex[]) =
        (run 16 1 (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sources (Some pcv) None (Some motifMem) None).[0]
    /// fs:788-822: greedy in-place sweeps (GIBBS_PHASE_MOTIF_GREEDY = 32)
    let findBestMotifPositionsWithStartPositionByPCV motifAmount motifLength pseudoCount cutOff alphabet sources (pcv:ProbabilityCompositeVector) (motifMem:MotifIndex[]) =
        (run 32 1 0UL motifAmount motifLength pseudoCount cutOff alphabet sources (Some pcv) None (Some motifMem) None).[0]
    /// fs:876-879
    let doMotifSamplingWithPCV motifAmount motifLength pseudoCount cutOff alphabet sources (pcv:ProbabilityCompositeVector) =
        (run 0 1 (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sources (Some pcv) None None None).[0]
    /// fs:1034-1038
    let doMotifSampling motifAmount motifLength pseudoCount cutOff alphabet sources =
        (run 0 1 (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sources None None None None).[0]
    /// fs:1028-1032
    let doMotifSamplingWithPPM motifAmount motifLength pseudoCount cutOff alphabet sources (ppM:PositionMatrix.PositionProbabilityMatrix) =
        (run 0 1 (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sources None (Some ppM) None None).[0]

    /// fs:856-881 / fs:973-998 / fs:1001-1026: numberOfRepetitions + 1 parallel restarts; the promote-or-restart loop is decided
    /// by the library (gibbs_fetch_best)
    let findBestInormationContentContainingMotifsWithPCV numberOfRepetitions motifAmount motifLength pseudoCount cutOff alphabet sources (pcv:ProbabilityCompositeVector) =
        (run 0 (numberOfRepetitions + 1) (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sources (Some pcv) None None (Some numberOfRepetitions)).[0]
    /// the script's second live call (fsx:407: reps 1, motifAmount 2, k 6, pc 1e-4, cutOff 1.0)
    let getMotifsWithBestInformationContents numberOfRepetitions motifAmount motifLength pseudoCount cutOff alphabet sources =
        (run 0 (numberOfRepetitions + 1) (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sources None None None (Some numberOfRepetitions)).[0]
    let getBestPWMSsOfPPM numberOfRepetitions motifAmount motifLength pseudoCount cutOff alphabet sources (ppM:PositionMatrix.PositionProbabilityMatrix) =
        (run 0 (numberOfRepetitions + 1) (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sources None (Some ppM) None (Some numberOfRepetitions)).[0]

    /// The restart loops of many sets in one batch over EVERY GPU of the box (gibbs_multi_batch_run_motif_device): set s gets
    /// exactly what the single-set call with the same seed gives (restart r of every set draws from the stream (seed, r)),
    /// whatever the number of devices; only the winners are copied back.
    let private bestOfSets (numberOfRepetitions:int) seed (motifAmount:int) k pc (cutOff:float) alphabet (sets:BioArray.BioArray<#IBioItem>[][])
                           (pcvs:ProbabilityCompositeVector[] option) : MotifIndex[][] =
        let m = max motifAmount 1
        let all = Array.concat sets
        let buf, offsets = Native.flatten all
        let setOffsets = Array.zeroCreate<int> (sets.Length + 1)
        sets |> Array.iteri (fun s src -> setOffsets.[s + 1] <- setOffsets.[s] + src.Length)
        let mutable b = IntPtr.Zero
        Native.check (Native.gibbs_multi_batch_create(buf, offsets, setOffsets, sets.Length, null, 0, &b))   // 0 = every visible device
        try
            let mutable p = Native.makeParams k pc alphabet (pcvs |> Option.map (fun v -> v.[0])) 0
            p.sampler <- 1; p.cutoff <- cutOff; p.motifAmount <- m
            let bg =
                match pcvs with
                | Some v -> v |> Array.collect (fun pcv -> [| for c in "ACGT" -> pcv.Array.[int c - 42] |])
                | None -> null
            Native.check (Native.gibbs_multi_batch_run_motif_device(b, &p, bg, numberOfRepetitions + 1, 0L, seed))
            let sites, scores, pos = Array.zeroCreate all.Length, Array.zeroCreate all.Length, Array.zeroCreate (all.Length * m)
            let nOut, restart = Array.zeroCreate sets.Length, Array.zeroCreate sets.Length
            let mutable stats = Native.GibbsRunStats()
            Native.check (Native.gibbs_multi_batch_fetch_best(b, numberOfRepetitions, sites, scores, nOut, null, restart, null, &stats))
            Native.check (Native.gibbs_multi_batch_fetch_best_positions(b, m, pos))
            Array.init sets.Length (fun s ->
                let o = setOffsets.[s]
                if restart.[s] < 0 then [| createMotifIndex 0. [] |]    // the loop's initial value survived
                else Array.init nOut.[s] (fun i -> createMotifIndex scores.[o + i] ([ for j in 0 .. m - 1 do
                                                                                         let q = pos.[(o + i) * m + j]
                                                                                         if q >= 0 then yield q ])))
        finally
            Native.gibbs_multi_batch_destroy b |> ignore

    /// findBestInormationContentContainingMotifsWithPCV of every set (pcvs.[s] the background of sets.[s]) in one batch over every GPU
    let findBestInormationContentContainingMotifsWithPCVOfSets numberOfRepetitions motifAmount motifLength pseudoCount cutOff alphabet sets (pcvs:ProbabilityCompositeVector[]) =
        bestOfSets numberOfRepetitions (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sets (Some pcvs)
    /// getMotifsWithBestInformationContents of every set in one batch over every GPU (e.g. the script's fsx:407 call per gene group)
    let getMotifsWithBestInformationContentsOfSets numberOfRepetitions motifAmount motifLength pseudoCount cutOff alphabet sets =
        bestOfSets numberOfRepetitions (seedOf None) motifAmount motifLength pseudoCount cutOff alphabet sets None
