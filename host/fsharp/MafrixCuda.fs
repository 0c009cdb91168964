// MafrixCuda.fs -- the reference-side binding of libmafrix_cuda (include/mafrix_cuda.h).
//
// SOURCE ONLY: there is no .NET SDK in the build image, so this file has never been compiled here.  It is the file a
// MafrixRender maintainer adds to EngineCore (after Core/Integrator/Integrators.fs in EngineCore.fsproj) to swap the
// CPU PixelIntegrator (Integrators.fs:141-172) for the GPU one; INTEGRATION.md walks through it.  Every struct is
// written into unmanaged memory by hand at the offsets tests/test_host_abi.py checks against the C header, so nothing
// depends on the CLR's struct marshalling rules.
module Engine.Core.MafrixCuda

open System
open System.Runtime.InteropServices
open Engine.Core.Color
open Engine.Core.Point
open Engine.Core.Texture
open Engine.Core.Camera
open Engine.Core.Light
open Engine.Core.Accels.BvhNode
open Engine.Core.Shapes.Triangle
open Engine.Core.Shapes.Rect
open Engine.Core.Shapes.Sphere
open Engine.Core.Interfaces.IIntegrator
open Engine.Core.Interfaces.IMaterial
open Engine.Core.Material

[<Struct; StructLayout(LayoutKind.Sequential)>]
type MfxSampleParams =                       // 40 bytes, include/mafrix_cuda.h: MfxSampleParams
    val mutable precision : int              // 0 = MFX_EXACT_F64 (bit-exact restatement), 1 = MFX_FAST_F32
    val mutable spp : int
    val mutable seed : uint64
    val mutable firstSample : int
    val mutable tileSize : int
    val mutable rank : int
    val mutable world : int
    val mutable flags : int                  // 2 = MFX_SAMPLE_REFERENCE_STREAM (rejection sampler on the exact stream),
                                             // 8 = MFX_SAMPLE_F32_PRIMARY (bounce 0 with f32 primitive tests instead of the id-exact kernel)

module Native =
    [<Literal>]
    let Lib = "mafrix_cuda"                  // libmafrix_cuda.so next to the executable / on LD_LIBRARY_PATH
    [<DllImport(Lib)>] extern int mfx_init(int device)
    [<DllImport(Lib)>] extern nativeint mfx_last_error()
    [<DllImport(Lib)>] extern int mfx_scene_create(nativeint desc, nativeint& scene)
    [<DllImport(Lib)>] extern int mfx_scene_destroy(nativeint scene)
    [<DllImport(Lib)>] extern int mfx_pixel_integrator_sample(nativeint scene, MfxSampleParams& p, nativeint texture)
    // Sample without the wait: frame k downloads while frame k+1 renders (two pinned textures, Film.fs:67-73's loop pipelined)
    [<DllImport(Lib)>] extern int mfx_pixel_integrator_sample_async(nativeint scene, MfxSampleParams& p, nativeint texture)
    [<DllImport(Lib)>] extern int mfx_pixel_integrator_wait(nativeint scene)
    // N GPUs behind this one render thread: the library replicates the scene and shards the frame by column stripes
    [<DllImport(Lib)>] extern int mfx_multi_create(nativeint desc, nativeint devices, int nDevices, nativeint& multi)
    [<DllImport(Lib)>] extern int mfx_multi_destroy(nativeint multi)
    [<DllImport(Lib)>] extern int mfx_multi_sample(nativeint multi, MfxSampleParams& p, nativeint texture)
    [<DllImport(Lib)>] extern int mfx_host_register(nativeint ptr, uint64 bytes)
    [<DllImport(Lib)>] extern int mfx_host_unregister(nativeint ptr)
    [<DllImport(Lib)>] extern int mfx_film_create(nativeint scene, nativeint& film)
    [<DllImport(Lib)>] extern int mfx_film_destroy(nativeint film)
    [<DllImport(Lib)>] extern int mfx_film_get_frame(nativeint film, MfxSampleParams& p, nativeint texture)
    [<DllImport(Lib)>] extern int mfx_film_post_process(nativeint film, nativeint rgba8)
    // the Film over the N GPUs of an mfx_multi handle: every device accumulates and tone-maps its own stripes
    [<DllImport(Lib)>] extern int mfx_multi_film_create(nativeint multi, nativeint& film)
    [<DllImport(Lib)>] extern int mfx_multi_film_destroy(nativeint film)
    [<DllImport(Lib)>] extern int mfx_multi_film_reset(nativeint film)
    [<DllImport(Lib)>] extern int mfx_multi_film_get_frame(nativeint film, MfxSampleParams& p, nativeint texture)
    [<DllImport(Lib)>] extern int mfx_multi_film_post_process(nativeint film, nativeint rgba8)
    [<DllImport(Lib)>] extern int mfx_multi_film_export(nativeint film, nativeint sum, double& frameCount)
    [<DllImport(Lib)>] extern int mfx_multi_film_import(nativeint film, nativeint sum, double frameCount)
    // the sphere sample (RenderTest/Sample/RayTracing.fs, MFX_SKY_TRACER): RayTraceCamera's constructor -> MfxLensCamera (152 B)
    [<DllImport(Lib)>] extern int mfx_camera_lens(double[] lookfrom, double[] lookat, double[] vup, double vfov, double aspect, double aperture, double focusDist, nativeint out)

let private check rc =
    if rc <> 0 then failwithf "libmafrix_cuda (%d): %s" rc (Marshal.PtrToStringAnsi(Native.mfx_last_error()))

/// Unmanaged images of the C structs.  Offsets: MfxPrim 104 B {kind@0, material@4, v[12]@8}; MfxMaterial 56 B
/// {kind@0, albedo@8, fuzz@32, ei@40, et@48}; MfxBvhNode 56 B {pmin@0, pmax@24, first@48, count@52};
/// MfxSceneDesc 320 B {prims@0, n@8, materials@16, n@24, nodes@32, n@40, indices@48, light@56, camera@200,
/// width@296, height@300, max_depth@304, integrator@308, sky@312 (NULL here: the sphere sample of
/// RenderTest/Sample/RayTracing.fs has no F# host types to marshal from -- its scene is built by the caller)}.
module private Interop =
    let inline wd (p:nativeint) (off:int) (v:float) = Marshal.WriteInt64(p, off, BitConverter.DoubleToInt64Bits v)
    let inline wpt (p:nativeint) (off:int) (q:Point) = wd p off q.x; wd p (off + 8) q.y; wd p (off + 16) q.z

    let prims (hs:IHitable[]) =
        let mem = Marshal.AllocHGlobal(104 * hs.Length)
        hs |> Array.iteri (fun i h ->
            let b = 104 * i
            for k in 0 .. 12 do Marshal.WriteInt64(mem, b + 8 * k, 0L)
            match h with                                                   // type tests as in Scene.fs:155-160
            | :? Triangle as t ->
                Marshal.WriteInt32(mem, b, 0); Marshal.WriteInt32(mem, b + 4, t.material)
                wpt mem (b + 8) t.v0; wpt mem (b + 32) t.v1; wpt mem (b + 56) t.v2
            | :? Rect as r ->                                              // Rect(p0,p1,p2,p3) = (p0,p1,p2) + (p0,p2,p3)
                Marshal.WriteInt32(mem, b, 1); Marshal.WriteInt32(mem, b + 4, r.trig1.material)
                wpt mem (b + 8) r.trig1.v0; wpt mem (b + 32) r.trig1.v1; wpt mem (b + 56) r.trig1.v2; wpt mem (b + 80) r.trig2.v2
            | :? Sphere as s ->
                Marshal.WriteInt32(mem, b, 2); Marshal.WriteInt32(mem, b + 4, s.material)
                wpt mem (b + 8) s.center; wd mem (b + 32) s.radius
            | _ -> failwith "CudaPixelIntegrator: unknown IHitable")
        mem

    /// quirk Q8: indices are global (IMaterial.fs:20-35) -> ship the table as it stands now.
    /// fuzz / ei / et are constructor arguments kept private in Material.fs:58,98: expose them (three one-line
    /// members) or pass them here; `props` returns (kind, fuzz, ei, et) for one IMaterial.
    let materials (ms:IMaterial[]) (props:IMaterial -> int * float * float * float) =
        let mem = Marshal.AllocHGlobal(56 * max 1 ms.Length)
        ms |> Array.iteri (fun i m ->
            let b = 56 * i
            let kind, fuzz, ei, et = props m
            let c = m.BaseColor()
            Marshal.WriteInt32(mem, b, kind); Marshal.WriteInt32(mem, b + 4, 0)
            wd mem (b + 8) c.r; wd mem (b + 16) c.g; wd mem (b + 24) c.b
            wd mem (b + 32) fuzz; wd mem (b + 40) ei; wd mem (b + 48) et)
        mem

    /// the tree exactly as Bvh.Build produced it, unstable sort and all (quirk Q9)
    let nodes (ns:BvhNode[]) =
        let mem = Marshal.AllocHGlobal(56 * ns.Length)
        ns |> Array.iteri (fun i n ->
            let b = 56 * i
            wpt mem b n.bound.pMin; wpt mem (b + 24) n.bound.pMax
            Marshal.WriteInt32(mem, b + 48, n.first); Marshal.WriteInt32(mem, b + 52, n.count))
        mem

    let ints (xs:int[]) =
        let mem = Marshal.AllocHGlobal(4 * max 1 xs.Length)
        Marshal.Copy(xs, 0, mem, xs.Length)
        mem

/// IPixelIntegrator over the GPU, built from the very objects Scene's constructor already has (Scene.fs:298-313).
type CudaPixelIntegrator(width:int, height:int, cam:PinholeCamera, bvh:Bvh, light:NewAreaLight, maxDepth:int,
                         materialProps:IMaterial -> int * float * float * float, ?newPathTracer:bool, ?fast:bool, ?seed:uint64, ?gpus:int) =
    let texture = Array2D.zeroCreate<Color> width height       // Color = 4 x float64, blittable; [x,y] at (x*h+y)*4
    let tex2d = new Texture2D<Color>(texture, width, height)
    let pin = GCHandle.Alloc(texture, GCHandleType.Pinned)      // pinned once + registered: the download is one DMA
    let mutable frame = 0
    let nGpus = defaultArg gpus 1                                // > 1: mfx_multi_* (devices 0 .. gpus-1), same single-threaded caller
    let scene =
        let mats = MaterialManager.GetManager().materials
        let pPrims, pMats = Interop.prims bvh.primitives, Interop.materials mats materialProps
        let pNodes, pIdx = Interop.nodes bvh.nodes, Interop.ints bvh.indices
        let d = Marshal.AllocHGlobal 320
        try
            Marshal.WriteIntPtr(d, 0, pPrims);  Marshal.WriteInt32(d, 8, bvh.primitives.Length)
            Marshal.WriteIntPtr(d, 16, pMats);  Marshal.WriteInt32(d, 24, mats.Length)
            Marshal.WriteIntPtr(d, 32, pNodes); Marshal.WriteInt32(d, 40, bvh.nodes.Length)
            Marshal.WriteIntPtr(d, 48, pIdx)
            let r = light.rect                                   // light: p0..p3, normal, colour (Light.fs:32-41)
            Interop.wpt d 56 r.trig1.v0; Interop.wpt d 80 r.trig1.v1; Interop.wpt d 104 r.trig1.v2; Interop.wpt d 128 r.trig2.v2
            Interop.wd d 152 light.normal.x; Interop.wd d 160 light.normal.y; Interop.wd d 168 light.normal.z
            Interop.wd d 176 light.color.r;  Interop.wd d 184 light.color.g;  Interop.wd d 192 light.color.b
            // camera as derived by the PinholeCamera constructor (Camera.fs:122-133; quirk Q5 stays on the host)
            Interop.wpt d 200 cam.position; Interop.wpt d 224 cam.topleft
            Interop.wd d 248 cam.coord.right.x; Interop.wd d 256 cam.coord.right.y; Interop.wd d 264 cam.coord.right.z
            Interop.wd d 272 cam.coord.down.x;  Interop.wd d 280 cam.coord.down.y;  Interop.wd d 288 cam.coord.down.z
            Marshal.WriteInt32(d, 296, width); Marshal.WriteInt32(d, 300, height)
            Marshal.WriteInt32(d, 304, maxDepth)
            Marshal.WriteInt32(d, 308, (if defaultArg newPathTracer false then 1 else 0))
            Marshal.WriteIntPtr(d, 312, 0n)                      // MfxSceneDesc.sky: only MFX_SKY_TRACER reads it
            check (Native.mfx_init 0)
            let mutable h = 0n
            if nGpus > 1 then check (Native.mfx_multi_create(d, 0n, nGpus, &h))   // one replica per device, Bvh shared
            else check (Native.mfx_scene_create(d, &h))          // copies everything: the buffers die right here
            check (Native.mfx_host_register(pin.AddrOfPinnedObject(), uint64 (width * height * 32)))
            h
        finally
            for p in [ d; pPrims; pMats; pNodes; pIdx ] do Marshal.FreeHGlobal p
    /// the scene handle (an MfxMulti when gpus > 1) and the params of the next n samples: fresh samples every displayed frame
    member this.Handle = scene
    member this.Gpus = nGpus
    member this.NextParams(n:int) =
        let mutable p = MfxSampleParams()
        p.precision <- (if defaultArg fast true then 1 else 0)
        p.spp <- n; p.seed <- defaultArg seed 1UL
        p.firstSample <- frame; p.world <- 1
        frame <- frame + n
        p
    interface IPixelIntegrator with
        member this.Sample(n:int) =                              // Integrators.fs:160-172
            let mutable p = this.NextParams n
            if nGpus > 1 then check (Native.mfx_multi_sample(scene, &p, pin.AddrOfPinnedObject()))   // every device DMAs its stripes
            else check (Native.mfx_pixel_integrator_sample(scene, &p, pin.AddrOfPinnedObject()))
            tex2d
    interface IDisposable with
        member this.Dispose() =
            Native.mfx_host_unregister(pin.AddrOfPinnedObject()) |> ignore
            (if nGpus > 1 then Native.mfx_multi_destroy scene else Native.mfx_scene_destroy scene) |> ignore
            pin.Free()

/// Film.GetFrame + PostProcessAndToScreenBuffer kept on the GPU(s) (Film.fs:18-34, Scene.fs:315-330).  The window loop of
/// Scene.Render (:331-333) becomes `film.GetFrame 1; film.PostProcess buffer`: only the RGBA8 screen crosses PCIe.  With
/// gpus > 1 every device keeps the Film of its own column stripes (mfx_multi_film_*), bit-identical to one GPU.
/// Dispose it before the integrator.
type CudaFilm(integrator:CudaPixelIntegrator) =
    let multi = integrator.Gpus > 1
    let film =
        let mutable h = 0n
        if multi then check (Native.mfx_multi_film_create(integrator.Handle, &h))
        else check (Native.mfx_film_create(integrator.Handle, &h))
        h
    /// Film.GetFrame(integrator, n): the target stays on the device(s)
    member this.GetFrame(n:int) =
        let mutable p = integrator.NextParams n
        if multi then check (Native.mfx_multi_film_get_frame(film, &p, 0n))
        else check (Native.mfx_film_get_frame(film, &p, 0n))
    /// PostProcessAndToScreenBuffer into the window's w*h*4 byte buffer
    member this.PostProcess(buffer:byte[]) =
        let pin = GCHandle.Alloc(buffer, GCHandleType.Pinned)
        try
            if multi then check (Native.mfx_multi_film_post_process(film, pin.AddrOfPinnedObject()))
            else check (Native.mfx_film_post_process(film, pin.AddrOfPinnedObject()))
        finally pin.Free()
    interface IDisposable with
        member this.Dispose() =
            (if multi then Native.mfx_multi_film_destroy film else Native.mfx_film_destroy film) |> ignore
