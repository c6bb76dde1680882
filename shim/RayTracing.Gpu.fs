// RayTracing.Gpu.fs — F# host-side binding of librtfs_b200.so for Smaug123/ray-tracing-fsharp.
//
// STATUS: source only.  This image has no .NET SDK (dotnet / fsc / mono are absent), so this file has
// NOT been compiled or run; it is the binding a maintainer would add, written against the reference's
// types as they are at RayTracing/*.fs.  The same marshalling, field for field, is exercised from
// Python (ray_tracing_fsharp_b200/domain.py `marshal`, native.py) by the test-suite.
//
// Where it goes: into the RayTracing project (RayTracing/RayTracing.fsproj), after Scene.fs in the
// compile order, because it reads the private records `Sphere` (Sphere.fs:302-310) and
// `InfinitePlane` (InfinitePlane.fs:101-106).  It adds `Scene.renderGpu`, with the signature of
// `Scene.render` (Scene.fs:196-204), over a `GpuScene` built by `GpuScene.make : Hittable array -> GpuScene`
// (the counterpart of `Scene.make`, Scene.fs:15-28), and `SceneGpu.renderWithProgress`, the same frame traced in passes
// with progress reported as they finish (a `GpuFrame`, rt_frame_*, for callers that want the passes themselves), and
// `SceneGpu.renderWithProgressUntil`, which also stops the frame once its per-pixel noise estimate is below a tolerance,
// and `SceneGpu.renderConverging`, which stops sampling each pixel once its own estimate is.
namespace RayTracing

open System
open System.Runtime.CompilerServices
open System.Runtime.InteropServices

#nowarn "9" // StructLayout / NativePtr

/// Mirrors of the structs of include/rtfs_b200.h (field order and types must match exactly).
module internal Native =

    [<Literal>]
    let Lib = "rtfs_b200" // librtfs_b200.so on the loader path

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtTexture =
        val mutable kind : int
        val mutable colourR : byte
        val mutable colourG : byte
        val mutable colourB : byte
        val mutable pad0 : byte
        val mutable width : int
        val mutable height : int
        val mutable rgb8 : nativeint
        val mutable even : int
        val mutable odd : int
        val mutable gridSize : float
        val mutable mapCentreX : float
        val mutable mapCentreY : float
        val mutable mapCentreZ : float
        val mutable mapRadius : float

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtHittable =
        val mutable shape : int
        val mutable style : int
        val mutable pX : float
        val mutable pY : float
        val mutable pZ : float
        val mutable nX : float
        val mutable nY : float
        val mutable nZ : float
        val mutable radius : float
        val mutable albedo : float
        val mutable fuzz : float
        val mutable ior : float
        val mutable prob : float
        val mutable texture : int
        val mutable colourR : byte
        val mutable colourG : byte
        val mutable colourB : byte
        val mutable pad0 : byte

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtCamera =
        val mutable viewOriginX : float
        val mutable viewOriginY : float
        val mutable viewOriginZ : float
        val mutable viewDirX : float
        val mutable viewDirY : float
        val mutable viewDirZ : float
        val mutable xAxisOriginX : float
        val mutable xAxisOriginY : float
        val mutable xAxisOriginZ : float
        val mutable xAxisDirX : float
        val mutable xAxisDirY : float
        val mutable xAxisDirZ : float
        val mutable yAxisDirX : float
        val mutable yAxisDirY : float
        val mutable yAxisDirZ : float
        val mutable viewportWidth : float
        val mutable viewportHeight : float
        val mutable focalLength : float
        val mutable samplesPerPixel : int
        val mutable bounceDepth : int

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtRenderOpts =
        val mutable seed : uint64
        val mutable adaptive : int
        val mutable mode : int
        val mutable gamma : int
        val mutable flags : int

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtStats =
        val mutable paths : uint64
        val mutable rays : uint64
        val mutable boxTests : uint64
        val mutable primTests : uint64
        val mutable kernelMs : float
        val mutable totalMs : float
        val mutable pixelsEarlyOut : uint64
        val mutable launches : int
        val mutable pad0 : int
        val mutable mainMs : float
        val mutable mainRays : uint64
        val mutable degeneratePaths : uint64

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtFrameProgress =
        val mutable samplesDone : int
        val mutable samplesTarget : int
        val mutable pathsDone : uint64
        val mutable pathsTarget : uint64
        val mutable pixelsFlagged : uint64
        val mutable lastPassMs : float
        val mutable deviceMs : float
        val mutable passes : int
        val mutable isDone : int // `done` in the header (a keyword in F#)

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtFrameNoise =
        val mutable pixels : uint64
        val mutable pixelsAbove : uint64
        val mutable maxSe : float
        val mutable meanSe : float
        val mutable tolerance : float

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtFrameConvergence =
        val mutable tolerance : float
        val mutable minSamples : int
        val mutable interval : int
        val mutable nextCheck : int
        val mutable checks : int
        val mutable pixelsActive : uint64
        val mutable pixelsConverged : uint64

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtDenoiseOpts =
        val mutable iterations : int
        val mutable featureSamples : int
        val mutable sigmaColour : float
        val mutable sigmaNormal : float
        val mutable sigmaAlbedo : float
        val mutable sigmaDepth : float
        val mutable gamma : int
        val mutable pad0 : int

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtSceneUpdate =
        val mutable objects : int
        val mutable textures : int
        val mutable spheresMoved : int
        val mutable nodesRefit : int
        val mutable generation : uint64
        val mutable deviceMs : float
        val mutable launches : int
        val mutable pad0 : int

    [<Struct ; StructLayout(LayoutKind.Sequential)>]
    type RtSceneRebuild =
        val mutable objectsRemoved : int
        val mutable objectsAppended : int
        val mutable nObjects : int
        val mutable nBounded : int
        val mutable nodes : int
        val mutable depth : int
        val mutable onDevice : int
        val mutable launches : int
        val mutable generation : uint64
        val mutable deviceMs : float


    [<DllImport(Lib)>]
    extern nativeint rt_last_error ()

    [<DllImport(Lib)>]
    extern int rt_device_count ()

    [<DllImport(Lib)>]
    extern int rt_scene_create (RtHittable[] objects, int nObjects, RtTexture[] textures, int nTextures, int device, nativeint& scene)

    [<DllImport(Lib)>]
    extern void rt_scene_destroy (nativeint scene)

    [<DllImport(Lib)>]
    extern int rt_scene_update (nativeint scene, int[] objectIndex, RtHittable[] objects, int nObjects, int[] textureIndex, RtTexture[] textures, int nTextures, RtSceneUpdate& info)

    [<DllImport(Lib)>]
    extern int rt_scene_rebuild (nativeint scene, int[] remove, int nRemove, RtHittable[] append, int nAppend, RtSceneRebuild& info)

    [<DllImport(Lib)>]
    extern int rt_render (nativeint scene, RtCamera& camera, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, byte[] rgbOut, nativeint sumsOut, RtStats& stats)

    // many views of one scene in one submission (include/rtfs_b200.h, rt_render_views); seeds may be null
    [<DllImport(Lib)>]
    extern int rt_render_views (nativeint scene, RtCamera[] cameras, uint64[] seeds, int nViews, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, byte[] rgbOut, nativeint sumsOut, RtStats& stats)

    // progressive frames on one device (include/rtfs_b200.h, rt_frame_*)
    [<DllImport(Lib)>]
    extern int rt_frame_begin (nativeint scene, RtCamera& camera, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, nativeint& frame, RtFrameProgress& progress)

    [<DllImport(Lib)>]
    extern int rt_frame_advance (nativeint frame, int maxSamples, float targetMs, RtFrameProgress& progress)

    [<DllImport(Lib)>]
    extern int rt_frame_read (nativeint frame, int gamma, byte[] rgbOut, nativeint sumsOut)

    [<DllImport(Lib)>]
    extern int rt_frame_extend (nativeint frame, int samplesPerPixel)

    [<DllImport(Lib)>]
    extern void rt_frame_destroy (nativeint frame)

    [<DllImport(Lib)>]
    extern int rt_frame_noise (nativeint frame, float tolerance, float32[] seOut, uint64[] sqOut, RtFrameNoise& summary)

    [<DllImport(Lib)>]
    extern int rt_frame_set_convergence (nativeint frame, float tolerance, int minSamples, int interval)

    [<DllImport(Lib)>]
    extern int rt_frame_convergence (nativeint frame, RtFrameConvergence& out)

    // progressive frames of a batch of views (include/rtfs_b200.h, rt_frame_begin_views; ABI 6 still: detect by the symbol)
    [<DllImport(Lib)>]
    extern int rt_frame_begin_views (nativeint scene, RtCamera[] cameras, uint64[] seeds, int nViews, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, nativeint& frame, RtFrameProgress& progress)

    [<DllImport(Lib)>]
    extern int rt_frame_view_noise (nativeint frame, float tolerance, [<Out>] RtFrameNoise[] perView)

    // denoised previews of progressive frames and their first-hit features (include/rtfs_b200.h, rt_frame_denoise; ABI 6
    // still: detect by the symbol)
    [<DllImport(Lib)>]
    extern int rt_frame_features (nativeint frame, int samples, [<Out>] int[] primOut, [<Out>] byte[] albedoOut, [<Out>] float32[] normalOut, [<Out>] float32[] depthOut)

    [<DllImport(Lib)>]
    extern int rt_frame_denoise (nativeint frame, RtDenoiseOpts& opts, [<Out>] byte[] rgbOut, [<Out>] float32[] linearOut)

    // a window of a frame, in one call or as a progressive frame (include/rtfs_b200.h, rt_render_window; ABI 6 still: detect
    // by the symbol)
    [<DllImport(Lib)>]
    extern int rt_render_window (nativeint scene, RtCamera& camera, int maxWidthCoord, int maxHeightCoord, int row0, int col0, int rows, int cols, RtRenderOpts& opts, byte[] rgbOut, nativeint sumsOut, RtStats& stats)

    [<DllImport(Lib)>]
    extern int rt_frame_begin_window (nativeint scene, RtCamera& camera, int maxWidthCoord, int maxHeightCoord, int row0, int col0, int rows, int cols, RtRenderOpts& opts, nativeint& frame, RtFrameProgress& progress)

    [<DllImport(Lib)>]
    extern int rt_frame_save (nativeint frame, byte[] out, unativeint cap, unativeint& len)

    [<DllImport(Lib)>]
    extern int rt_frame_resume (nativeint scene, byte[] snapshot, unativeint len, nativeint& frame, RtFrameProgress& progress)

    [<DllImport(Lib)>]
    extern int rt_multi_frame_resume (nativeint multi, byte[] snapshot, unativeint len, nativeint& frame, RtFrameProgress& progress)

    [<DllImport(Lib)>]
    extern int rt_pixel_noise (int[] sums, uint64[] sq, unativeint n, float32[] seOut)

    [<DllImport(Lib)>]
    extern int rt_multi_create (RtHittable[] objects, int nObjects, RtTexture[] textures, int nTextures, int[] devices, int nDevices, nativeint& multi)

    [<DllImport(Lib)>]
    extern int rt_multi_render (nativeint multi, RtCamera& camera, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, byte[] rgbOut, nativeint sumsOut, RtStats& stats)

    [<DllImport(Lib)>]
    extern void rt_multi_destroy (nativeint multi)

    [<DllImport(Lib)>]
    extern int rt_multi_frame_begin (nativeint multi, RtCamera& camera, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, nativeint& frame, RtFrameProgress& progress)

    // a batch of views split over the devices of an RtMulti, in one call or as a progressive frame (include/rtfs_b200.h,
    // rt_multi_render_views; ABI 6 still: detect by the symbol)
    [<DllImport(Lib)>]
    extern int rt_multi_render_views (nativeint multi, RtCamera[] cameras, uint64[] seeds, int nViews, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, byte[] rgbOut, nativeint sumsOut, RtStats& stats)

    [<DllImport(Lib)>]
    extern int rt_multi_frame_begin_views (nativeint multi, RtCamera[] cameras, uint64[] seeds, int nViews, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, nativeint& frame, RtFrameProgress& progress)

    // one rank of a one-process-per-GPU job: the library issues the NCCL collectives itself (include/rtfs_b200.h, rt_comm_*)
    [<DllImport(Lib)>]
    extern int rt_comm_unique_id (byte[] idOut)

    [<DllImport(Lib)>]
    extern int rt_comm_create (byte[] id, int rank, int world, int device, nativeint stream, nativeint& comm)

    [<DllImport(Lib)>]
    extern int rt_comm_render (nativeint comm, nativeint scene, RtCamera& camera, int maxWidthCoord, int maxHeightCoord, RtRenderOpts& opts, byte[] rgbOut, nativeint sumsOut, RtStats& stats)

    [<DllImport(Lib)>]
    extern void rt_comm_destroy (nativeint comm)

    let check (rc : int) : unit =
        if rc <> 0 then
            failwithf "librtfs_b200 error %i: %s" rc (Marshal.PtrToStringAnsi (rt_last_error ()))

/// `ParameterisedTexture.toTexture` erases an image / checker texture to a closure (Texture.fs:69-72), which
/// cannot cross the ABI.  `GpuTexture.ofParameterised` builds the same `Texture` and remembers its structure,
/// keyed by the closure object, so that `GpuScene.make` can recover it.
[<RequireQualifiedAccess>]
module GpuTexture =
    let private table =
        ConditionalWeakTable<obj, (float * Point * ParameterisedTexture)> ()

    /// Drop-in for `ParameterisedTexture.toTexture (Sphere.planeMapInverse radius centre) texture`.
    let ofParameterised (radius : float) (centre : Point) (texture : ParameterisedTexture) : Texture =
        let t =
            ParameterisedTexture.toTexture (Sphere.planeMapInverse radius centre) texture

        match t with
        | Texture.Arbitrary f -> table.Add (box f, (radius, centre, texture))
        | Texture.Colour _ -> ()

        t

    /// Samples a `ParameterisedTexture` (typically an `Arbitrary` closure, which cannot run on the GPU) into an
    /// `Image` of `width` x `height` texels.  Texel (x, y) of an Image answers the lookups with
    /// `int ((1 - u) (W - 1)) = x` and `int (v (H - 1)) = y` (Texture.fs:63-67); it receives the texture's value
    /// at the centre of that cell.  An approximation by construction, hence explicit (same as
    /// `ParameterisedTexture.bake` in the Python mirror, domain.py).
    let bake (radius : float) (centre : Point) (width : int) (height : int) (texture : ParameterisedTexture) : ParameterisedTexture =
        let interpret = Sphere.planeMapInverse radius centre

        Array.init
            height
            (fun y ->
                let v = min 1.0 ((float y + 0.5) / float (height - 1))

                Array.init
                    width
                    (fun x ->
                        let u = max 0.0 (1.0 - (float x + 0.5) / float (width - 1))
                        ParameterisedTexture.colourAt interpret texture (Sphere.planeMap radius centre u v)
                    )
            )
        |> ParameterisedTexture.Image

    let internal tryStructure (t : Texture) : (float * Point * ParameterisedTexture) voption =
        match t with
        | Texture.Colour _ -> ValueNone
        | Texture.Arbitrary f ->
            match table.TryGetValue (box f) with
            | true, v -> ValueSome v
            | false, _ ->
                failwith
                    "GPU backend: Texture.Arbitrary is a host closure; build it with GpuTexture.ofParameterised (closures inside it: GpuTexture.bake)"

type GpuScene =
    private
        {
            Handle : nativeint
            IsMulti : bool
            Pins : GCHandle list
            /// the records the scene was made or last updated from, and each image texture's texels (null for the other
            /// kinds): SceneGpu.update diffs the new records against them
            mutable Hittables : Native.RtHittable[]
            mutable Textures : Native.RtTexture[]
            mutable Texels : byte[][]
        }

    interface IDisposable with
        member this.Dispose () =
            if this.IsMulti then
                Native.rt_multi_destroy this.Handle
            else
                Native.rt_scene_destroy this.Handle

            for p in this.Pins do
                p.Free ()

[<RequireQualifiedAccess>]
module GpuScene =

    let private setPoint (Point (struct (x, y, z))) (h : byref<Native.RtHittable>) =
        h.pX <- x
        h.pY <- y
        h.pZ <- z

    /// Flattens `ParameterisedTexture` into the texture table (children before parents, as domain.py does).
    let rec private addTexture
        (textures : ResizeArray<Native.RtTexture>)
        (pins : ResizeArray<GCHandle>)
        (radius : float)
        (Point (struct (cx, cy, cz)))
        (t : ParameterisedTexture)
        : int
        =
        let mutable e = Native.RtTexture ()
        e.even <- -1
        e.odd <- -1
        e.mapCentreX <- cx
        e.mapCentreY <- cy
        e.mapCentreZ <- cz
        e.mapRadius <- radius

        match t with
        | ParameterisedTexture.Colour p ->
            e.kind <- 0
            e.colourR <- p.Red
            e.colourG <- p.Green
            e.colourB <- p.Blue
        | ParameterisedTexture.Image img ->
            // img.[y].[x], rows already flipped by ofImage (Texture.fs:30-48): copy as row-major RGB8
            let h, w = img.Length, img.[0].Length
            let bytes = Array.zeroCreate<byte> (3 * w * h)

            for y in 0 .. h - 1 do
                for x in 0 .. w - 1 do
                    let p = img.[y].[x]
                    bytes.[3 * (y * w + x)] <- p.Red
                    bytes.[3 * (y * w + x) + 1] <- p.Green
                    bytes.[3 * (y * w + x) + 2] <- p.Blue

            let pin = GCHandle.Alloc (bytes, GCHandleType.Pinned)
            pins.Add pin
            e.kind <- 1
            e.width <- w
            e.height <- h
            e.rgb8 <- pin.AddrOfPinnedObject ()
        | ParameterisedTexture.Checkered (even, odd, gridSize) ->
            e.kind <- 2
            e.even <- addTexture textures pins radius (Point (struct (cx, cy, cz))) even
            e.odd <- addTexture textures pins radius (Point (struct (cx, cy, cz))) odd
            e.gridSize <- gridSize
        | ParameterisedTexture.Arbitrary _ ->
            failwith "GPU backend: ParameterisedTexture.Arbitrary is a host closure; bake it to an Image first"

        textures.Add e
        textures.Count - 1

    let private setTexture
        (textures : ResizeArray<Native.RtTexture>)
        (pins : ResizeArray<GCHandle>)
        (t : Texture)
        (h : byref<Native.RtHittable>)
        =
        h.texture <- -1

        match t with
        | Texture.Colour p ->
            h.colourR <- p.Red
            h.colourG <- p.Green
            h.colourB <- p.Blue
        | Texture.Arbitrary _ ->
            match GpuTexture.tryStructure t with
            | ValueSome (radius, centre, structure) -> h.texture <- addTexture textures pins radius centre structure
            | ValueNone -> ()

    let private setColour (p : Pixel) (h : byref<Native.RtHittable>) =
        h.texture <- -1
        h.colourR <- p.Red
        h.colourG <- p.Green
        h.colourB <- p.Blue

    /// The FloatProducer each material carries (Sphere.fs:21-37) is ignored: the device RNG is keyed per
    /// (seed, pixel, sample, bounce).
    let private marshalSphere textures pins (shape : int) (s : Sphere) : Native.RtHittable =
        let mutable h = Native.RtHittable ()
        h.shape <- shape
        setPoint s.Centre &h
        h.radius <- s.Radius

        match s.Style with
        | SphereStyle.LightSource tex ->
            h.style <- 0
            setTexture textures pins tex &h
        | SphereStyle.LightSourceCap colour ->
            h.style <- 1
            setColour colour &h
        | SphereStyle.PureReflection (albedo, tex) ->
            h.style <- 2
            h.albedo <- float albedo
            setTexture textures pins tex &h
        | SphereStyle.FuzzedReflection (albedo, tex, fuzz, _) ->
            h.style <- 3
            h.albedo <- float albedo
            h.fuzz <- float fuzz
            setTexture textures pins tex &h
        | SphereStyle.LambertReflection (albedo, tex, _) ->
            h.style <- 4
            h.albedo <- float albedo
            setTexture textures pins tex &h
        | SphereStyle.Dielectric (albedo, tex, ior, prob, _) ->
            h.style <- 5
            h.albedo <- float albedo
            h.ior <- float ior
            h.prob <- float prob
            setTexture textures pins tex &h
        | SphereStyle.Glass (albedo, tex, ior, _) ->
            h.style <- 6
            h.albedo <- float albedo
            h.ior <- float ior
            setTexture textures pins tex &h

        h

    let private marshalPlane textures pins (p : InfinitePlane) : Native.RtHittable =
        let mutable h = Native.RtHittable ()
        h.shape <- 2
        setPoint p.Point &h
        let (UnitVector (Vector (struct (nx, ny, nz)))) = p.Normal
        h.nX <- nx
        h.nY <- ny
        h.nZ <- nz

        match p.Style with
        | InfinitePlaneStyle.LightSource tex ->
            h.style <- 0
            setTexture textures pins tex &h
        | InfinitePlaneStyle.PureReflection (albedo, colour) ->
            h.style <- 2
            h.albedo <- float albedo
            setColour colour &h
        | InfinitePlaneStyle.FuzzedReflection (albedo, colour, fuzz, _) ->
            h.style <- 3
            h.albedo <- float albedo
            h.fuzz <- float fuzz
            setColour colour &h
        | InfinitePlaneStyle.LambertReflection (albedo, colour, _) ->
            h.style <- 4
            h.albedo <- float albedo
            setColour colour &h

        h

    /// The Hittable and texture records of `objects`, each image texture's texels (null for the other kinds), and the pins
    /// that hold the texels in place while the library copies them.
    let internal marshal (objects : Hittable array) =
        let textures = ResizeArray<Native.RtTexture> ()
        let pins = ResizeArray<GCHandle> ()

        let hittables =
            objects
            |> Array.map (fun o ->
                match o with
                | Hittable.Sphere s -> marshalSphere textures pins 0 s
                | Hittable.UnboundedSphere s -> marshalSphere textures pins 1 s
                | Hittable.InfinitePlane p -> marshalPlane textures pins p
            )

        let texels =
            textures.ToArray ()
            |> Array.map (fun t ->
                if t.kind = 1 then
                    pins |> Seq.find (fun p -> p.AddrOfPinnedObject () = t.rgb8) |> fun p -> p.Target :?> byte[]
                else
                    null
            )

        hittables, textures.ToArray (), texels, pins

    /// Counterpart of Scene.make (Scene.fs:15-28).  `devices`: CUDA ordinals; more than one splits every frame.
    let makeOn (devices : int[]) (objects : Hittable array) : GpuScene =
        let hittables, textures, texels, pins = marshal objects

        let texArr =
            if textures.Length = 0 then Array.zeroCreate 1 else textures

        let mutable handle = 0n

        if devices.Length > 1 then
            Native.rt_multi_create (hittables, hittables.Length, texArr, textures.Length, devices, devices.Length, &handle)
            |> Native.check
        else
            Native.rt_scene_create (hittables, hittables.Length, texArr, textures.Length, devices.[0], &handle)
            |> Native.check

        // the library copies everything it needs during create, so the pins can be released straight away
        for p in pins do
            p.Free ()

        {
            Handle = handle
            IsMulti = devices.Length > 1
            Pins = []
            Hittables = hittables
            Textures = textures
            Texels = texels
        }

    let make (objects : Hittable array) : GpuScene = makeOn [| 0 |] objects

/// What SceneGpu.update changed (RtSceneUpdate, include/rtfs_b200.h).
type SceneUpdate =
    {
        /// object records that changed
        Objects : int
        /// texture records that changed
        Textures : int
        /// bounded spheres whose device sphere (FP32 centre, radius) changed
        SpheresMoved : int
        /// tree nodes whose child boxes were recomputed
        NodesRefit : int
        /// the scene's edit count after the call (0 = as made)
        Generation : uint64
        /// device time of the copy and the kernels (CUDA events)
        DeviceMs : float
    }

/// What SceneGpu.addObjects, removeObjects and rebuild did (RtSceneRebuild, include/rtfs_b200.h).
type SceneRebuild =
    {
        /// objects taken out and added at the end
        ObjectsRemoved : int
        ObjectsAppended : int
        /// the scene's objects after the call, and the spheres in its tree
        Objects : int
        Bounded : int
        /// nodes and depth (internal nodes on the longest path) of the new tree
        Nodes : int
        Depth : int
        /// true: built on the device; false: the host SAH tree (the device tree was deeper than the walk stacks allow)
        OnDevice : bool
        /// the scene's edit count after the call
        Generation : uint64
        /// device time of the build (CUDA events)
        DeviceMs : float
    }

/// RtRenderOpts.flags bits a caller may pass to SceneGpu.openFrameWith (include/rtfs_b200.h, RT_FLAG_*).
[<RequireQualifiedAccess>]
module FrameFlags =
    /// RT_FLAG_NOISE: the frame also keeps the per-pixel sum of squares its noise estimate (GpuFrame.Noise) needs
    [<Literal>]
    let Noise = 128

/// The noise estimate of a progressive frame over the pixels later passes still sample (RtFrameNoise of
/// include/rtfs_b200.h, copied out of the native struct): how many there are, how many have a standard error of the mean
/// above the tolerance (8-bit levels), the largest and the mean standard error, and the tolerance asked for.
type FrameNoise =
    {
        Pixels : uint64
        PixelsAbove : uint64
        MaxSe : float
        MeanSe : float
        Tolerance : float
    }

/// The convergence rule of a progressive frame and its state (RtFrameConvergence of include/rtfs_b200.h): the tolerance
/// (8-bit levels), the checkpoints MinSamples + j * Interval, the next one, the checks run so far, the pixels still being
/// sampled and those a check has stopped.
type FrameConvergence =
    {
        Tolerance : float
        MinSamples : int
        Interval : int
        NextCheck : int
        Checks : int
        PixelsActive : uint64
        PixelsConverged : uint64
    }

/// A frame in progress on a GpuScene (rt_frame_*; on a multi-GPU scene split over its devices, bit for bit the frame of one
/// GPU): advanced in passes over windows of sample indices.
/// After every pass it is exactly the frame rt_render gives at `SamplesDone` samples per pixel with the same seed, so
/// `Read` shows the image sharpening; a caller stops early by not advancing any more, and `Extend` continues a finished
/// frame to more samples.  Dispose it before its scene.  A frame of a batch of views (SceneGpu.openFrameViews) holds `Views`
/// images of Rows * Cols pixels one after the other; the progress and convergence counts are sums over them.  A frame of a
/// window (SceneGpu.openFrameWindow) has the window's Rows and Cols, and its counts cover the window's pixels.
/// First-hit features of a progressive frame (GpuFrame.Features), row-major per view.
type FrameFeatures =
    {
        Prim : int[]
        Albedo : byte[]
        Normal : float32[]
        Depth : float32[]
    }

/// The options of GpuFrame.Denoise (RtDenoiseOpts; the formulas are in include/rtfs_b200.h).
type DenoiseOptions =
    {
        Iterations : int
        FeatureSamples : int
        SigmaColour : float
        SigmaNormal : float
        SigmaAlbedo : float
        SigmaDepth : float
    }

[<RequireQualifiedAccess>]
module DenoiseOptions =
    /// the suggested options (DESIGN.md section 19)
    let defaults : DenoiseOptions =
        {
            Iterations = 3
            FeatureSamples = 4
            SigmaColour = 4.0
            SigmaNormal = 0.1
            SigmaAlbedo = 16.0
            SigmaDepth = 0.02
        }

type GpuFrame internal (handle : nativeint, rows : int, cols : int, views : int, first : Native.RtFrameProgress) =
    let mutable handle = handle
    let mutable progress = first

    let noise (s : Native.RtFrameNoise) : FrameNoise =
        {
            Pixels = s.pixels
            PixelsAbove = s.pixelsAbove
            MaxSe = s.maxSe
            MeanSe = s.meanSe
            Tolerance = s.tolerance
        }

    member _.Rows = rows
    member _.Cols = cols
    member _.Views = views
    member _.SamplesDone = progress.samplesDone
    member _.SamplesTarget = progress.samplesTarget
    /// traceOnce calls so far, and in the whole frame (exact from the start)
    member _.PathsDone = progress.pathsDone
    member _.PathsTarget = progress.pathsTarget
    member _.LastPassMs = progress.lastPassMs
    member _.Passes = progress.passes
    member _.IsDone = progress.isDone <> 0

    /// One pass of at most `maxSamples` sample indices (0: no limit) sized to take about `targetMs` of device time
    /// (0: no limit).  Nothing happens once the frame is done.
    member _.Advance (maxSamples : int, targetMs : float) : unit =
        let mutable p = Native.RtFrameProgress ()
        Native.rt_frame_advance (handle, maxSamples, targetMs, &p) |> Native.check
        progress <- p

    /// The current image as row-major RGB8, 3 * Rows * Cols bytes per view (PixelOutput.correct applied when `gamma`).
    member _.Read (gamma : bool) : byte[] =
        let rgb = Array.zeroCreate<byte> (3 * views * rows * cols)
        Native.rt_frame_read (handle, (if gamma then 1 else 0), rgb, 0n) |> Native.check
        rgb

    /// The frame as a snapshot (rt_frame_save): bytes SceneGpu.resumeFrame opens again as this frame, in this process or
    /// another, on one GPU or several.  The frame is left as it was; a frame whose scene was edited since it opened fails.
    member _.Save () : byte[] =
        let mutable len = 0un
        Native.rt_frame_save (handle, null, 0un, &len) |> Native.check
        let out = Array.zeroCreate<byte> (int len)
        Native.rt_frame_save (handle, out, len, &len) |> Native.check
        out

    /// Sets the target to `samplesPerPixel`; fails if that would change the probe already run (firstTrial) or is below
    /// what the frame holds.
    member _.Extend (samplesPerPixel : int) : unit =
        Native.rt_frame_extend (handle, samplesPerPixel) |> Native.check

    /// The noise estimate of a frame opened with FrameFlags.Noise (rt_frame_noise): the summary over the pixels later
    /// passes still sample, against `tolerance` (8-bit levels), and with `wantMap` the standard error of every pixel,
    /// row-major Rows * Cols per view (null otherwise).
    member _.Noise (tolerance : float, wantMap : bool) : FrameNoise * float32[] =
        let map = if wantMap then Array.zeroCreate<float32> (views * rows * cols) else null
        let mutable summary = Native.RtFrameNoise ()
        Native.rt_frame_noise (handle, tolerance, map, null, &summary) |> Native.check
        noise summary, map

    /// One summary per view (rt_frame_view_noise): view v's pixels still being sampled, exactly `Noise`'s summary of the
    /// frame of that view alone.  Pixels = 0: the view is finished.
    member _.ViewNoise (tolerance : float) : FrameNoise[] =
        let out = Array.zeroCreate<Native.RtFrameNoise> views
        Native.rt_frame_view_noise (handle, tolerance, out) |> Native.check
        out |> Array.map noise

    /// Stops sampling each pixel once its standard error is within `tolerance` (8-bit levels), checked at the sample
    /// counts minSamples + j * interval (rt_frame_set_convergence).  Only on a frame opened with FrameFlags.Noise, before
    /// its first pass.  Every pixel is then exactly rt_render's pixel at the sample count it stopped at.
    member _.SetConvergence (tolerance : float, minSamples : int, interval : int) : unit =
        Native.rt_frame_set_convergence (handle, tolerance, minSamples, interval) |> Native.check

    /// First-hit features of sample indices 0 .. samples - 1 of every pixel (rt_frame_features), row-major per view: the
    /// Hittable index hit by sample 0 (-1: a miss); the truncating mean RGB8 of the colour the first scatter leaves in a white
    /// path; the mean shading normal (xyz) and the mean hit distance (+inf: no sample hit) over the samples that hit.  Exact
    /// functions of (seed, pixel, samples): passes do not change them.
    member _.Features (samples : int) : FrameFeatures =
        let n = views * rows * cols
        let prim = Array.zeroCreate<int> n
        let albedo = Array.zeroCreate<byte> (3 * n)
        let normal = Array.zeroCreate<float32> (3 * n)
        let depth = Array.zeroCreate<float32> n
        Native.rt_frame_features (handle, samples, prim, albedo, normal, depth) |> Native.check
        { Prim = prim ; Albedo = albedo ; Normal = normal ; Depth = depth }

    /// A denoised preview of the current image (rt_frame_denoise) as row-major RGB8 per view (PixelOutput.correct applied
    /// when `gamma`), leaving the frame as it was.  Only on a frame opened with FrameFlags.Noise.  DenoiseOptions.defaults
    /// holds the suggested options (DESIGN.md section 19).
    member _.Denoise (options : DenoiseOptions, gamma : bool) : byte[] =
        let rgb = Array.zeroCreate<byte> (3 * views * rows * cols)
        let mutable o = Native.RtDenoiseOpts ()
        o.iterations <- options.Iterations
        o.featureSamples <- options.FeatureSamples
        o.sigmaColour <- options.SigmaColour
        o.sigmaNormal <- options.SigmaNormal
        o.sigmaAlbedo <- options.SigmaAlbedo
        o.sigmaDepth <- options.SigmaDepth
        o.gamma <- (if gamma then 1 else 0)
        Native.rt_frame_denoise (handle, &o, rgb, null) |> Native.check
        rgb

    /// The rule set by SetConvergence and its state (rt_frame_convergence).
    member _.Convergence () : FrameConvergence =
        let mutable c = Native.RtFrameConvergence ()
        Native.rt_frame_convergence (handle, &c) |> Native.check

        {
            Tolerance = c.tolerance
            MinSamples = c.minSamples
            Interval = c.interval
            NextCheck = c.nextCheck
            Checks = c.checks
            PixelsActive = c.pixelsActive
            PixelsConverged = c.pixelsConverged
        }

    interface IDisposable with
        member _.Dispose () =
            Native.rt_frame_destroy handle
            handle <- 0n

[<RequireQualifiedAccess>]
module SceneGpu =

    let private marshalCamera (c : Camera) : Native.RtCamera =
        let mutable n = Native.RtCamera ()
        let (Point (struct (ox, oy, oz))) = Ray.origin c.View
        let (UnitVector (Vector (struct (vx, vy, vz)))) = Ray.vector c.View
        let (Point (struct (xox, xoy, xoz))) = Ray.origin c.ViewportXAxis
        let (UnitVector (Vector (struct (xx, xy, xz)))) = Ray.vector c.ViewportXAxis
        let (UnitVector (Vector (struct (yx, yy, yz)))) = Ray.vector c.ViewportYAxis
        n.viewOriginX <- ox
        n.viewOriginY <- oy
        n.viewOriginZ <- oz
        n.viewDirX <- vx
        n.viewDirY <- vy
        n.viewDirZ <- vz
        n.xAxisOriginX <- xox
        n.xAxisOriginY <- xoy
        n.xAxisOriginZ <- xoz
        n.xAxisDirX <- xx
        n.xAxisDirY <- xy
        n.xAxisDirZ <- xz
        n.yAxisDirX <- yx
        n.yAxisDirY <- yy
        n.yAxisDirZ <- yz
        n.viewportWidth <- c.ViewportWidth
        n.viewportHeight <- c.ViewportHeight
        n.focalLength <- c.FocalLength
        n.samplesPerPixel <- c.SamplesPerPixel
        n.bounceDepth <- c.BounceDepth
        n

    /// Same signature and laziness as Scene.render (Scene.fs:196-236): nothing is traced until a row is forced;
    /// the first forced row renders the whole frame on the GPU; every row reports progress once (Scene.fs:232).
    let render
        (progressIncrement : float<progress> -> unit)
        (_print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (camera : Camera)
        (s : GpuScene)
        : float<progress> * Image
        =
        let rowsIter = 2 * maxHeightCoord + 1
        let colsIter = 2 * maxWidthCoord + 1

        let frame =
            lazy
                (let rgb = Array.zeroCreate<byte> (3 * rowsIter * colsIter)
                 let mutable cam = marshalCamera camera
                 let mutable opts = Native.RtRenderOpts ()
                 // FloatProducer (Random ()) in the reference (Scene.fs:205): a fresh seed per frame
                 opts.seed <- uint64 (Random().NextInt64 ())
                 opts.adaptive <- 1
                 let mutable stats = Native.RtStats ()

                 if s.IsMulti then
                     Native.rt_multi_render (s.Handle, &cam, maxWidthCoord, maxHeightCoord, &opts, rgb, 0n, &stats)
                     |> Native.check
                 else
                     Native.rt_render (s.Handle, &cam, maxWidthCoord, maxHeightCoord, &opts, rgb, 0n, &stats)
                     |> Native.check

                 rgb)

        let rows =
            Seq.init
                rowsIter
                (fun row ->
                    async {
                        let rgb = frame.Force ()

                        let result =
                            Array.init
                                colsIter
                                (fun col ->
                                    let i = 3 * (row * colsIter + col)

                                    {
                                        Red = rgb.[i]
                                        Green = rgb.[i + 1]
                                        Blue = rgb.[i + 2]
                                    }
                                )

                        progressIncrement 1.0<progress>
                        return result
                    }
                )

        1.0<progress> * float rowsIter, Image.make rowsIter colsIter rows

    /// Scene.render for every camera of `cameras` (same SamplesPerPixel and BounceDepth; a turntable, a fly-through,
    /// stereo pairs, previews), rendered together in one rt_render_views call, or on a multi-GPU scene one
    /// rt_multi_render_views call split over its devices (bit for bit the batch of one GPU): one Image per camera, lazy
    /// like `render` (the first forced row of any view renders them all).  Every row of every view reports progress once:
    /// rows * cameras.Length in all.  One fresh seed per view, as `render` draws one per frame.
    let renderViews
        (progressIncrement : float<progress> -> unit)
        (_print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (cameras : Camera array)
        (s : GpuScene)
        : float<progress> * Image array
        =
        let rowsIter = 2 * maxHeightCoord + 1
        let colsIter = 2 * maxWidthCoord + 1
        let n = cameras.Length

        let frames =
            lazy
                (let rgb = Array.zeroCreate<byte> (3 * rowsIter * colsIter * n)
                 let cams = cameras |> Array.map marshalCamera
                 let seeds = Array.init n (fun _ -> uint64 (Random().NextInt64 ()))
                 let mutable opts = Native.RtRenderOpts ()
                 opts.adaptive <- 1
                 let mutable stats = Native.RtStats ()

                 if s.IsMulti then
                     Native.rt_multi_render_views (s.Handle, cams, seeds, n, maxWidthCoord, maxHeightCoord, &opts, rgb, 0n, &stats)
                     |> Native.check
                 else
                     Native.rt_render_views (s.Handle, cams, seeds, n, maxWidthCoord, maxHeightCoord, &opts, rgb, 0n, &stats)
                     |> Native.check

                 rgb)

        let image (view : int) =
            let rows =
                Seq.init
                    rowsIter
                    (fun row ->
                        async {
                            let rgb = frames.Force ()
                            let start = 3 * ((view * rowsIter + row) * colsIter)

                            let result =
                                Array.init
                                    colsIter
                                    (fun col ->
                                        let i = start + 3 * col

                                        {
                                            Red = rgb.[i]
                                            Green = rgb.[i + 1]
                                            Blue = rgb.[i + 2]
                                        }
                                    )

                            progressIncrement 1.0<progress>
                            return result
                        }
                    )

            Image.make rowsIter colsIter rows

        1.0<progress> * float (rowsIter * n), Array.init n image

    /// The window (row0, col0, rows, cols) of `render`'s image, traced without the rest of the frame (rt_render_window) on a
    /// single-device scene: a closer look at one part of a frame, or one tile of a frame split between processes.  Lazy like
    /// `render`; every row of the window reports progress once.  `seed` is the frame's: windows of one seed are crops of one
    /// frame, bit for bit, so tiles of any grid reassemble into it.
    let renderWindow
        (progressIncrement : float<progress> -> unit)
        (_print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (camera : Camera)
        (row0 : int, col0 : int, rowsIter : int, colsIter : int)
        (seed : uint64)
        (s : GpuScene)
        : float<progress> * Image
        =
        if s.IsMulti then
            failwith "GPU backend: a window runs on a single-device GpuScene"

        let frame =
            lazy
                (let rgb = Array.zeroCreate<byte> (3 * rowsIter * colsIter)
                 let mutable cam = marshalCamera camera
                 let mutable opts = Native.RtRenderOpts ()
                 opts.seed <- seed
                 opts.adaptive <- 1
                 let mutable stats = Native.RtStats ()

                 Native.rt_render_window (s.Handle, &cam, maxWidthCoord, maxHeightCoord, row0, col0, rowsIter, colsIter, &opts, rgb, 0n, &stats)
                 |> Native.check

                 rgb)

        let rows =
            Seq.init
                rowsIter
                (fun row ->
                    async {
                        let rgb = frame.Force ()

                        let result =
                            Array.init
                                colsIter
                                (fun col ->
                                    let i = 3 * (row * colsIter + col)

                                    {
                                        Red = rgb.[i]
                                        Green = rgb.[i + 1]
                                        Blue = rgb.[i + 2]
                                    }
                                )

                        progressIncrement 1.0<progress>
                        return result
                    }
                )

        1.0<progress> * float rowsIter, Image.make rowsIter colsIter rows

    /// Opens a progressive frame with RtRenderOpts.flags `flags` (e.g. FrameFlags.Noise for GpuFrame.Noise).  On a
    /// multi-GPU scene the frame is split over its devices (rt_multi_frame_begin) and is bit for bit the frame of one GPU.
    let openFrameWith (flags : int) (maxWidthCoord : int) (maxHeightCoord : int) (camera : Camera) (seed : uint64) (s : GpuScene) : GpuFrame =
        let mutable cam = marshalCamera camera
        let mutable opts = Native.RtRenderOpts ()
        opts.seed <- seed
        opts.adaptive <- 1
        opts.flags <- flags
        let mutable handle = 0n
        let mutable progress = Native.RtFrameProgress ()

        let rc =
            if s.IsMulti then
                Native.rt_multi_frame_begin (s.Handle, &cam, maxWidthCoord, maxHeightCoord, &opts, &handle, &progress)
            else
                Native.rt_frame_begin (s.Handle, &cam, maxWidthCoord, maxHeightCoord, &opts, &handle, &progress)

        Native.check rc

        new GpuFrame (handle, 2 * maxHeightCoord + 1, 2 * maxWidthCoord + 1, 1, progress)

    /// Opens a progressive frame (rt_frame_begin, or rt_multi_frame_begin on a multi-GPU scene: the probe runs now).
    let openFrame (maxWidthCoord : int) (maxHeightCoord : int) (camera : Camera) (seed : uint64) (s : GpuScene) : GpuFrame =
        openFrameWith 0 maxWidthCoord maxHeightCoord camera seed s

    /// Opens a progressive frame of a batch of views (rt_frame_begin_views: the probe of every view runs now) with
    /// RtRenderOpts.flags `flags`: `cameras` with the same SamplesPerPixel and BounceDepth, one seed per view.  View v is
    /// exactly the frame openFrameWith gives for cameras.[v] and seeds.[v].  On a multi-GPU scene the frame is split over
    /// its devices (rt_multi_frame_begin_views) and is bit for bit the frame of one GPU.
    let openFrameViews (flags : int) (maxWidthCoord : int) (maxHeightCoord : int) (cameras : Camera array) (seeds : uint64 array) (s : GpuScene) : GpuFrame =
        if seeds.Length <> cameras.Length then
            invalidArg "seeds" "one seed per camera"

        let cams = cameras |> Array.map marshalCamera
        let mutable opts = Native.RtRenderOpts ()
        opts.adaptive <- 1
        opts.flags <- flags
        let mutable handle = 0n
        let mutable progress = Native.RtFrameProgress ()

        let rc =
            if s.IsMulti then
                Native.rt_multi_frame_begin_views (s.Handle, cams, seeds, cams.Length, maxWidthCoord, maxHeightCoord, &opts, &handle, &progress)
            else
                Native.rt_frame_begin_views (s.Handle, cams, seeds, cams.Length, maxWidthCoord, maxHeightCoord, &opts, &handle, &progress)

        Native.check rc

        new GpuFrame (handle, 2 * maxHeightCoord + 1, 2 * maxWidthCoord + 1, cameras.Length, progress)

    /// Opens a progressive frame of the window (row0, col0, rows, cols) of the frame openFrameWith gives (rt_frame_begin_window:
    /// the probe of the window's pixels runs now) with RtRenderOpts.flags `flags`.  Its Rows and Cols are the window's, and
    /// after every pass (under a convergence rule too) it is exactly that crop of the frame openFrameWith gives for the same
    /// camera and seed.  Single-device scenes only.
    let openFrameWindow (flags : int) (maxWidthCoord : int) (maxHeightCoord : int) (camera : Camera) (row0 : int, col0 : int, rows : int, cols : int) (seed : uint64) (s : GpuScene) : GpuFrame =
        if s.IsMulti then
            failwith "GPU backend: a progressive frame of a window runs on a single-device GpuScene"

        let mutable cam = marshalCamera camera
        let mutable opts = Native.RtRenderOpts ()
        opts.seed <- seed
        opts.adaptive <- 1
        opts.flags <- flags
        let mutable handle = 0n
        let mutable progress = Native.RtFrameProgress ()

        Native.rt_frame_begin_window (s.Handle, &cam, maxWidthCoord, maxHeightCoord, row0, col0, rows, cols, &opts, &handle, &progress)
        |> Native.check

        new GpuFrame (handle, rows, cols, 1, progress)

    /// Opens a progressive frame from a snapshot written by GpuFrame.Save (rt_frame_resume, or rt_multi_frame_resume on a
    /// multi-GPU scene).  After every further pass it is bit for bit the saved frame continued without interruption,
    /// whatever device count saved it.  The scene must hold the objects and textures of the saved frame's scene; a window
    /// resumes on a single-device scene only.  The frame's shape is read from the snapshot's header (RtSnapshotHeader).
    let resumeFrame (s : GpuScene) (snapshot : byte[]) : GpuFrame =
        let mutable handle = 0n
        let mutable progress = Native.RtFrameProgress ()

        let rc =
            if s.IsMulti then
                Native.rt_multi_frame_resume (s.Handle, snapshot, unativeint snapshot.Length, &handle, &progress)
            else
                Native.rt_frame_resume (s.Handle, snapshot, unativeint snapshot.Length, &handle, &progress)

        Native.check rc
        // RtSnapshotHeader: kind at byte 48, n_views at 52, max_width_coord / max_height_coord at 208 / 212, window rows and
        // cols at 224 / 228
        let i32 (at : int) = System.BitConverter.ToInt32 (snapshot, at)
        let kind, views = i32 48, i32 52
        let rows, cols = if kind = 2 then i32 224, i32 228 else 2 * i32 212 + 1, 2 * i32 208 + 1
        new GpuFrame (handle, rows, cols, views, progress)

    /// The scene GpuScene.make would give for `objects` (the whole new object list), made in place on the device
    /// (rt_scene_update): the list is marshalled and diffed against the scene's current records, and only the changed objects
    /// and textures are sent; the device refits the tree.  The scene then renders bit for bit as GpuScene.make objects.  The
    /// structure must stay (the object count, each object's shape, the sign of each bounded sphere's radius, the texture
    /// table's size, kinds and image sizes); a structural change fails, as does a multi-GPU scene.  Frames opened before the
    /// call are stale: GpuFrame.Advance and the calls that trace fail on them.
    let update (s : GpuScene) (objects : Hittable array) : SceneUpdate =
        if s.IsMulti then
            failwith "GPU backend: SceneGpu.update edits a single-device GpuScene; make a multi-GPU scene anew"

        let hittables, textures, texels, pins = GpuScene.marshal objects

        try
            let sameShape (a : Native.RtTexture) (b : Native.RtTexture) =
                a.kind = b.kind && (a.kind <> 1 || (a.width = b.width && a.height = b.height))

            if hittables.Length <> s.Hittables.Length
               || textures.Length <> s.Textures.Length
               || not (Array.forall2 sameShape textures s.Textures) then
                failwith "GPU backend: SceneGpu.update keeps the scene's structure (object count, texture table); make a new scene"

            let sameTexture (j : int) =
                let a, b = textures.[j], s.Textures.[j]

                a.kind = b.kind && a.colourR = b.colourR && a.colourG = b.colourG && a.colourB = b.colourB
                && a.even = b.even && a.odd = b.odd && a.gridSize = b.gridSize && a.mapCentreX = b.mapCentreX
                && a.mapCentreY = b.mapCentreY && a.mapCentreZ = b.mapCentreZ && a.mapRadius = b.mapRadius
                && (a.kind <> 1 || texels.[j] = s.Texels.[j])

            let objectIndex =
                [| for i in 0 .. hittables.Length - 1 do
                       if hittables.[i] <> s.Hittables.[i] then
                           yield i |]

            let textureIndex =
                [| for j in 0 .. textures.Length - 1 do
                       if not (sameTexture j) then
                           yield j |]

            let mutable info = Native.RtSceneUpdate ()
            // the pins hold the new texels in place until the call returns (the library copies them)
            Native.rt_scene_update (
                s.Handle,
                objectIndex,
                Array.map (fun i -> hittables.[i]) objectIndex,
                objectIndex.Length,
                textureIndex,
                Array.map (fun j -> textures.[j]) textureIndex,
                textureIndex.Length,
                &info
            )
            |> Native.check

            s.Hittables <- hittables
            s.Textures <- textures
            s.Texels <- texels

            {
                Objects = info.objects
                Textures = info.textures
                SpheresMoved = info.spheresMoved
                NodesRefit = info.nodesRefit
                Generation = info.generation
                DeviceMs = info.deviceMs
            }
        finally
            for p in pins do
                p.Free ()

    let private restructure (s : GpuScene) (remove : int array) (append : Native.RtHittable array) : SceneRebuild =
        if s.IsMulti then
            failwith "GPU backend: structural edits change a single-device GpuScene; make a multi-GPU scene anew"

        let mutable info = Native.RtSceneRebuild ()

        Native.rt_scene_rebuild (s.Handle, remove, remove.Length, append, append.Length, &info)
        |> Native.check

        let gone = Set.ofArray remove

        s.Hittables <-
            Array.append
                [| for i in 0 .. s.Hittables.Length - 1 do
                       if not (gone.Contains i) then
                           yield s.Hittables.[i] |]
                append

        {
            ObjectsRemoved = info.objectsRemoved
            ObjectsAppended = info.objectsAppended
            Objects = info.nObjects
            Bounded = info.nBounded
            Nodes = info.nodes
            Depth = info.depth
            OnDevice = info.onDevice <> 0
            Generation = info.generation
            DeviceMs = info.deviceMs
        }

    /// Appends `objects` to the scene in place (rt_scene_rebuild): the device builds the tree anew, and the scene then renders
    /// bit for bit as GpuScene.make of its objects followed by these.  Their textures must be textures the scene already
    /// holds (the texture table cannot grow here); otherwise, and on a multi-GPU scene, the call fails.  Frames opened before
    /// the call are stale.
    let addObjects (s : GpuScene) (objects : Hittable array) : SceneRebuild =
        let hittables, textures, texels, pins = GpuScene.marshal objects

        try
            let find (j : int) =
                let a = textures.[j]

                s.Textures
                |> Array.tryFindIndex (fun b ->
                    a.kind = b.kind && a.colourR = b.colourR && a.colourG = b.colourG && a.colourB = b.colourB
                    && a.even = b.even && a.odd = b.odd && a.gridSize = b.gridSize && a.mapCentreX = b.mapCentreX
                    && a.mapCentreY = b.mapCentreY && a.mapCentreZ = b.mapCentreZ && a.mapRadius = b.mapRadius
                    && a.width = b.width && a.height = b.height)
                |> Option.filter (fun k -> a.kind <> 1 || texels.[j] = s.Texels.[k])
                |> Option.defaultWith (fun () ->
                    failwith "GPU backend: SceneGpu.addObjects: an object brings a texture the scene does not hold; make a new scene")

            let remap = Array.init textures.Length find

            let appended =
                hittables
                |> Array.map (fun h ->
                    let mutable h = h
                    if h.texture >= 0 then h.texture <- remap.[h.texture]
                    h)

            restructure s [||] appended
        finally
            for p in pins do
                p.Free ()

    /// Removes the objects at `indices` in place (rt_scene_rebuild): the others keep their order and are renumbered densely,
    /// and the scene renders bit for bit as GpuScene.make of them.  Bad or repeated indices, or a multi-GPU scene, fail.
    /// Frames opened before the call are stale.
    let removeObjects (s : GpuScene) (indices : int array) : SceneRebuild = restructure s indices [||]

    /// Builds the scene's tree anew on the device from its current objects: the remedy for a tree that update's refits have
    /// left slow to walk (DESIGN.md section 20).  Frames are unchanged bit for bit; frames opened before the call are stale.
    let rebuild (s : GpuScene) : SceneRebuild = restructure s [||] [||]

    // the frame of renderWithProgressUntil and renderConverging: passes of about 250 ms with progress ticks, an optional
    // convergence rule (tolerance, minSamples, interval) and an optional stop on the noise summary (tolerance, fraction)
    let private renderInPasses
        (rule : (float * int * int) option)
        (noiseStop : (float * float) option)
        (progressIncrement : float<progress> -> unit)
        (_print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (camera : Camera)
        (s : GpuScene)
        : float<progress> * Image
        =
        let rowsIter = 2 * maxHeightCoord + 1
        let colsIter = 2 * maxWidthCoord + 1

        let frame =
            lazy
                (let flags = if noiseStop.IsSome || rule.IsSome then FrameFlags.Noise else 0

                 use f =
                    openFrameWith flags maxWidthCoord maxHeightCoord camera (uint64 (Random().NextInt64 ())) s

                 match rule with
                 | Some (tolerance, minSamples, interval) -> f.SetConvergence (tolerance, minSamples, interval)
                 | None -> ()

                 let ticked = ref 0

                 // ticks so far = floor(rows * pathsDone / pathsTarget): the fraction carries to the next pass
                 let tick () =
                     let want =
                         if f.IsDone || f.PathsTarget = 0UL then
                             rowsIter
                         else
                             min rowsIter (int (float rowsIter * float f.PathsDone / float f.PathsTarget))

                     for _ in ticked.Value + 1 .. want do
                         progressIncrement 1.0<progress>

                     ticked.Value <- max ticked.Value want

                 let converged () =
                     match noiseStop with
                     | Some (tolerance, fraction) when not f.IsDone ->
                         let summary, _ = f.Noise (tolerance, false)
                         float summary.PixelsAbove <= fraction * float summary.Pixels
                     | _ -> false

                 tick ()
                 let mutable stop = converged ()

                 while not f.IsDone && not stop do
                     f.Advance (0, 250.0)
                     tick ()
                     stop <- converged ()

                 // a frame stopped on its noise hands out the rest of the rows' ticks
                 for _ in ticked.Value + 1 .. rowsIter do
                     progressIncrement 1.0<progress>

                 ticked.Value <- rowsIter
                 f.Read false)

        let rows =
            Seq.init
                rowsIter
                (fun row ->
                    async {
                        let rgb = frame.Force ()

                        return
                            Array.init
                                colsIter
                                (fun col ->
                                    let i = 3 * (row * colsIter + col)

                                    {
                                        Red = rgb.[i]
                                        Green = rgb.[i + 1]
                                        Blue = rgb.[i + 2]
                                    }
                                )
                    }
                )

        1.0<progress> * float rowsIter, Image.make rowsIter colsIter rows

    /// `renderWithProgress` with a stop on the noise estimate: with `Some (tolerance, fraction)` the frame stops at the
    /// first check (after the probe, then after every pass) where at most `fraction` of the pixels still being sampled
    /// have a standard error of the mean above `tolerance` (8-bit levels); the image is then rt_render's at the samples
    /// done.  `None` is renderWithProgress.
    let renderWithProgressUntil
        (noiseStop : (float * float) option)
        (progressIncrement : float<progress> -> unit)
        (print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (camera : Camera)
        (s : GpuScene)
        : float<progress> * Image
        =
        renderInPasses None noiseStop progressIncrement print maxWidthCoord maxHeightCoord camera s

    /// `renderWithProgress` where each pixel stops being sampled once its standard error of the mean is within
    /// `tolerance` (8-bit levels), checked at minSamples + j * interval samples (GpuFrame.SetConvergence, e.g. 64 and 64):
    /// every pixel is rt_render's pixel at the sample count it stopped at, and smooth regions cost fewer paths.
    let renderConverging
        (tolerance : float, minSamples : int, interval : int)
        (progressIncrement : float<progress> -> unit)
        (print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (camera : Camera)
        (s : GpuScene)
        : float<progress> * Image
        =
        renderInPasses (Some (tolerance, minSamples, interval)) None progressIncrement print maxWidthCoord maxHeightCoord camera s

    /// `render`'s signature and laziness, but the frame is traced in passes of about 250 ms of device time and
    /// `progressIncrement 1.0<progress>` is called as passes finish, in proportion to the paths traced out of the frame's
    /// total: `rows` calls in all, as the reference makes (Scene.fs:232).  A multi-GPU scene splits every pass over its devices.
    let renderWithProgress
        (progressIncrement : float<progress> -> unit)
        (print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (camera : Camera)
        (s : GpuScene)
        : float<progress> * Image
        =
        renderWithProgressUntil None progressIncrement print maxWidthCoord maxHeightCoord camera s

    /// `renderViews` traced as one converging progressive frame of the batch (openFrameViews): passes of about 250 ms of
    /// device time advance every view, and each pixel stops being sampled once its standard error of the mean is within
    /// `tolerance` (8-bit levels), checked at minSamples + j * interval samples.  View v is exactly `renderConverging`'s
    /// image of cameras.[v] with the same seed and rule; a batch pays each pass's fixed cost once instead of once per view.
    /// rows * cameras.Length progress calls in all, as passes finish.  One fresh seed per view.
    let renderViewsConverging
        (tolerance : float, minSamples : int, interval : int)
        (progressIncrement : float<progress> -> unit)
        (_print : string -> unit)
        (maxWidthCoord : int)
        (maxHeightCoord : int)
        (cameras : Camera array)
        (s : GpuScene)
        : float<progress> * Image array
        =
        let rowsIter = 2 * maxHeightCoord + 1
        let colsIter = 2 * maxWidthCoord + 1
        let n = cameras.Length
        let total = rowsIter * n

        let frames =
            lazy
                (let seeds = Array.init n (fun _ -> uint64 (Random().NextInt64 ()))
                 use f = openFrameViews FrameFlags.Noise maxWidthCoord maxHeightCoord cameras seeds s
                 f.SetConvergence (tolerance, minSamples, interval)
                 let ticked = ref 0

                 let tick () =
                     let want =
                         if f.IsDone || f.PathsTarget = 0UL then
                             total
                         else
                             min total (int (float total * float f.PathsDone / float f.PathsTarget))

                     for _ in ticked.Value + 1 .. want do
                         progressIncrement 1.0<progress>

                     ticked.Value <- max ticked.Value want

                 tick ()

                 while not f.IsDone do
                     f.Advance (0, 250.0)
                     tick ()

                 f.Read false)

        let image (view : int) =
            let rows =
                Seq.init
                    rowsIter
                    (fun row ->
                        async {
                            let rgb = frames.Force ()
                            let start = 3 * ((view * rowsIter + row) * colsIter)

                            return
                                Array.init
                                    colsIter
                                    (fun col ->
                                        let i = start + 3 * col

                                        {
                                            Red = rgb.[i]
                                            Green = rgb.[i + 1]
                                            Blue = rgb.[i + 2]
                                        }
                                    )
                        }
                    )

            Image.make rowsIter colsIter rows

        1.0<progress> * float total, Array.init n image
