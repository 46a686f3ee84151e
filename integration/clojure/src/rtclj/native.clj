(ns rtclj.native
  "One downcall into librtclj_b200.so (include/rtclj_b200.h) in place of the render loops of
   raytracing/-main (src/raytracing.clj:141-171) and realm.raytracing/-main
   (src/realm/raytracing.clj:325-346).  JDK >= 22 (java.lang.foreign).
   UNEXECUTED in the build image (no JVM there); the same ABI is exercised from Python and from a
   plain-C client, and tests/test_clojure_binding.py checks every byte offset written in `layouts`
   below against the C header (ctypes offsetof / sizeof), so this file cannot drift from it."
  (:import [java.lang.foreign Arena FunctionDescriptor Linker Linker$Option MemoryLayout
            MemorySegment SymbolLookup ValueLayout]))

(def ^:private ^Linker linker (Linker/nativeLinker))
(def ^:private lib (SymbolLookup/libraryLookup "librtclj_b200.so" (Arena/global)))

(defn- downcall [^String sym ^FunctionDescriptor fd]
  (.downcallHandle linker (.orElseThrow (.find lib sym)) fd (make-array Linker$Option 0)))

;; ---- struct layouts of include/rtclj_b200.h: {:size bytes :fields {field byte-offset}}
;; BEGIN-LAYOUTS (parsed by tests/test_clojure_binding.py)
(def layouts
  {:rtclj_scene  {:size 56
                  :fields {:n 0 :center_xyz 8 :radius 16 :material 24 :albedo_rgb 32 :fuzz 40 :ior 48}}
   :rtclj_camera {:size 160
                  :fields {:pixel00 0 :pixel_du 24 :pixel_dv 48 :center 72 :defocus_u 96 :defocus_v 120
                           :defocus_angle 144 :width 152 :height 156}}
   :rtclj_params {:size 48
                  :fields {:spp 0 :max_depth 4 :seed 8 :flags 16 :samples_per_unit 20 :shard_index 24
                           :shard_count 28 :shard_rows 32 :device 36}}
   :rtclj_stats  {:size 72
                  :fields {:samples 0 :segments 8 :exact_tests 16 :list_overflows 24 :prefilter_tests 32
                           :device_ms 40 :kernel_ms 48 :total_ms 56 :samples_per_unit 64 :n_devices 68}}})
;; END-LAYOUTS

(defn- off ^long [struct field] (long (get-in layouts [struct :fields field])))
(defn- size ^long [struct] (long (get-in layouts [struct :size])))

(defn- fd-int [& args]
  (FunctionDescriptor/of ValueLayout/JAVA_INT (into-array MemoryLayout args)))

;; int rtclj_render(const rtclj_scene*, const rtclj_camera*, const rtclj_params*,
;;                  double* out_linear, uint8_t* out_rgb8, rtclj_stats*)
(def ^:private rtclj-render
  (downcall "rtclj_render" (apply fd-int (repeat 6 ValueLayout/ADDRESS))))
;; int rtclj_render_multi(const rtclj_scene*, const rtclj_camera*, const rtclj_params*,
;;                        const int32_t* devices, int32_t n_devices,
;;                        double* out_linear, uint8_t* out_rgb8, rtclj_stats*)
(def ^:private rtclj-render-multi
  (downcall "rtclj_render_multi"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS)))
;; int rtclj_render_frames(const rtclj_scene*, const rtclj_camera* cameras, int32_t n_frames,
;;                         const rtclj_params*, const int32_t* devices, int32_t n_devices,
;;                         double* out_linear, uint8_t* out_rgb8, rtclj_stats*)
(def ^:private rtclj-render-frames
  (downcall "rtclj_render_frames"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS)))
;; int rtclj_render_multi_ppm(const rtclj_scene*, const rtclj_camera*, const rtclj_params*,
;;                            const int32_t* devices, int32_t n_devices,
;;                            char* out, size_t capacity, size_t* len, rtclj_stats*)
(def ^:private rtclj-render-multi-ppm
  (downcall "rtclj_render_multi_ppm"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_LONG ValueLayout/ADDRESS
                    ValueLayout/ADDRESS)))
;; int rtclj_render_multi_png(const rtclj_scene*, const rtclj_camera*, const rtclj_params*,
;;                            const int32_t* devices, int32_t n_devices,
;;                            uint8_t* out, size_t capacity, size_t* len, rtclj_stats*)
(def ^:private rtclj-render-multi-png
  (downcall "rtclj_render_multi_png"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_LONG ValueLayout/ADDRESS
                    ValueLayout/ADDRESS)))
;; int rtclj_host_alloc(size_t bytes, void** out);  int rtclj_host_free(void* p)
(def ^:private rtclj-host-alloc (downcall "rtclj_host_alloc" (fd-int ValueLayout/JAVA_LONG ValueLayout/ADDRESS)))
(def ^:private rtclj-host-free (downcall "rtclj_host_free" (fd-int ValueLayout/ADDRESS)))
;; const char* rtclj_last_error(void)
(def ^:private rtclj-last-error
  (downcall "rtclj_last_error" (FunctionDescriptor/of ValueLayout/ADDRESS (make-array MemoryLayout 0))))

(def flags-main  (bit-or 1 2 4 8)) ; near-zero guard | Schlick | innermost-first product | sum / spp
(def flags-realm 0)
(def flags-i     (bit-or 16 32))   ; normal shading | int(255.999 c)

(defn- doubles-seg ^MemorySegment [^Arena a xs]
  (.allocateFrom a ValueLayout/JAVA_DOUBLE (double-array xs)))

(defn- last-error ^String []
  (let [^MemorySegment p (.invokeWithArguments rtclj-last-error [])]
    (.getString (.reinterpret p 512) 0)))

(defn- check! [rc]
  (when-not (zero? (int rc))
    (throw (ex-info (last-error) {:rtclj/code (int rc)}))))

(defn- pinned-doubles
  "W*H*3 doubles of PINNED host memory (rtclj_host_alloc): the GPUs write the image into it
   directly, without the library's staging copy.  Returns [segment free-fn]."
  [^Arena a ^long n-doubles]
  (let [slot (.allocate a 8 8)
        _    (check! (.invokeWithArguments rtclj-host-alloc [(* 8 n-doubles) slot]))
        ^MemorySegment p (.reinterpret (.get slot ValueLayout/ADDRESS 0) (* 8 n-doubles))]
    [p #(.invokeWithArguments rtclj-host-free [p])]))

(defn- fill-camera!
  "Writes the camera map `cam` (see `render`) into the rtclj_camera at `camera`."
  [^MemorySegment camera cam]
  (let [put3 (fn [field ^doubles v]
               (dotimes [k 3]
                 (.set camera ValueLayout/JAVA_DOUBLE (+ (off :rtclj_camera field) (* 8 k)) (aget v k))))]
    (put3 :pixel00 (:pixel-00-loc cam)) (put3 :pixel_du (:pixel-du cam))
    (put3 :pixel_dv (:pixel-dv cam)) (put3 :center (:camera-center cam))
    (put3 :defocus_u (:defocus-disk-u cam)) (put3 :defocus_v (:defocus-disk-v cam))
    (.set camera ValueLayout/JAVA_DOUBLE (off :rtclj_camera :defocus_angle) (double (:defocus-angle cam)))
    (.set camera ValueLayout/JAVA_INT (off :rtclj_camera :width) (int (:image-width cam)))
    (.set camera ValueLayout/JAVA_INT (off :rtclj_camera :height) (int (:image-height cam)))
    camera))

(defn- marshal
  "Fills rtclj_scene / rtclj_camera / rtclj_params in arena `a`; returns [scene camera params]."
  [^Arena a bodies cam samples-per-px max-depth {:keys [seed flags device samples-per-unit]
                                                 :or {seed 1 flags flags-main device 0 samples-per-unit 0}}]
  (let [scene  (doto (.allocate a (size :rtclj_scene) 8)
                 (.set ValueLayout/JAVA_INT (off :rtclj_scene :n) (int (count bodies)))
                 (.set ValueLayout/ADDRESS (off :rtclj_scene :center_xyz) (doubles-seg a (mapcat :rtclj/center bodies)))
                 (.set ValueLayout/ADDRESS (off :rtclj_scene :radius) (doubles-seg a (map :rtclj/radius bodies)))
                 (.set ValueLayout/ADDRESS (off :rtclj_scene :material)
                       (.allocateFrom a ValueLayout/JAVA_INT (int-array (map :rtclj/kind bodies))))
                 (.set ValueLayout/ADDRESS (off :rtclj_scene :albedo_rgb) (doubles-seg a (mapcat :rtclj/albedo bodies)))
                 (.set ValueLayout/ADDRESS (off :rtclj_scene :fuzz) (doubles-seg a (map :rtclj/fuzz bodies)))
                 (.set ValueLayout/ADDRESS (off :rtclj_scene :ior) (doubles-seg a (map :rtclj/ior bodies))))
        camera (fill-camera! (.allocate a (size :rtclj_camera) 8) cam)
        params (doto (.allocate a (size :rtclj_params) 8)
                 (.set ValueLayout/JAVA_INT (off :rtclj_params :spp) (int samples-per-px))
                 (.set ValueLayout/JAVA_INT (off :rtclj_params :max_depth) (int max-depth))
                 (.set ValueLayout/JAVA_LONG (off :rtclj_params :seed) (long seed))
                 (.set ValueLayout/JAVA_INT (off :rtclj_params :flags) (int flags))
                 (.set ValueLayout/JAVA_INT (off :rtclj_params :samples_per_unit) (int samples-per-unit))
                 (.set ValueLayout/JAVA_INT (off :rtclj_params :device) (int device)))]
    [scene camera params]))

(defn render
  "bodies : hittable list made with rtclj.scene, in LIST ORDER (the first body wins a tie).
   cam    : {:pixel-00-loc :pixel-du :pixel-dv :camera-center :defocus-disk-u :defocus-disk-v
            :defocus-angle :image-width :image-height} -- the locals of raytracing.clj:105-139,
            each vector a double[3].
   :devices [0 1 .. 7] interleaves the image rows over several GPUs from this one process
   (rtclj_render_multi; the reference's pool, raytracing.clj:157-171); default: GPU 0.
   :samples-per-unit n  sums n samples sequentially per work unit.  Default 0 = the library chooses:
   the reference's strict order (one sequential sum per pixel, raytracing.clj:142-155) for primary-ray
   renders, whose contract is bit-exactness, and chunks of ~27 samples added in index order for
   full-depth renders (<= 1e-13 relative difference; north_star allows 1e-3).  Pass samples-per-px
   to force the strict order everywhere: the library then buffers every sample's colour in HBM and adds
   them in sample order, 2 % slower than chunks on one B200 and 6 % on eight -- DESIGN.md section 4.5.
   Returns a vector of double[3] (linear RGB), row-major from the top-left pixel, i.e. `colors`
   of raytracing.clj:170-171, ready for the existing write-color! loop (:172-175)."
  [bodies cam samples-per-px max-depth & {:keys [devices] :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [w      (long (:image-width cam))
          h      (long (:image-height cam))
          [scene camera params] (marshal a bodies cam samples-per-px max-depth opts)
          [^MemorySegment out free!] (pinned-doubles a (* 3 w h))]
      (try
        (check!
         (if (seq devices)
           (.invokeWithArguments rtclj-render-multi
                                 [scene camera params
                                  (.allocateFrom a ValueLayout/JAVA_INT (int-array devices)) (int (count devices))
                                  out MemorySegment/NULL MemorySegment/NULL])
           (.invokeWithArguments rtclj-render
                                 [scene camera params out MemorySegment/NULL MemorySegment/NULL])))
        (mapv (fn [^long p]
                (double-array [(.getAtIndex out ValueLayout/JAVA_DOUBLE (* 3 p))
                               (.getAtIndex out ValueLayout/JAVA_DOUBLE (+ 1 (* 3 p)))
                               (.getAtIndex out ValueLayout/JAVA_DOUBLE (+ 2 (* 3 p)))]))
              (range (* w h)))
        (finally (free!))))))

(defn render-frames
  "A camera sequence of one scene (rtclj_render_frames): `cams` is a seq of camera maps (see `render`) of one image
   size -- a turntable, a fly-through, a focus pull.  All frames share the GPU launches (one kernel tail per launch
   instead of one per frame); frame f is bit-identical to (render bodies (nth cams f) ...) with the same options,
   which `render` takes as well (:devices, :seed, :flags, :samples-per-unit).  One seed for every frame.  Returns a
   vector with one frame per camera, each frame what `render` returns."
  [bodies cams samples-per-px max-depth & {:keys [devices] :or {devices [0]} :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [cam0    (first cams)
          w       (long (:image-width cam0))
          h       (long (:image-height cam0))
          k       (count cams)
          [scene _ params] (marshal a bodies cam0 samples-per-px max-depth opts)
          cameras (.allocate a (* k (size :rtclj_camera)) 8)
          _       (doseq [[i cam] (map-indexed vector cams)]
                    (fill-camera! (.asSlice cameras (* i (size :rtclj_camera)) (size :rtclj_camera)) cam))
          [^MemorySegment out free!] (pinned-doubles a (* 3 w h k))]
      (try
        (check! (.invokeWithArguments rtclj-render-frames
                                      [scene cameras (int k) params
                                       (.allocateFrom a ValueLayout/JAVA_INT (int-array devices)) (int (count devices))
                                       out MemorySegment/NULL MemorySegment/NULL]))
        (mapv (fn [^long f]
                (mapv (fn [^long p]
                        (let [q (* 3 (+ p (* f w h)))]
                          (double-array [(.getAtIndex out ValueLayout/JAVA_DOUBLE q)
                                         (.getAtIndex out ValueLayout/JAVA_DOUBLE (+ 1 q))
                                         (.getAtIndex out ValueLayout/JAVA_DOUBLE (+ 2 q))])))
                      (range (* w h))))
              (range k))
        (finally (free!))))))

(defn render-ppm!
  "Everything between the camera let-block and ppm->png in raytracing/-main (raytracing.clj:141-175) as ONE
   native call: the render loop on :devices (default [0]) and the write-color! loop on the first of them;
   the text of scene.ppm comes back and is handed to a single .write.  The image never visits the host."
  [^String path bodies cam samples-per-px max-depth & {:keys [devices] :or {devices [0]} :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [w    (long (:image-width cam))
          h    (long (:image-height cam))
          [scene camera params] (marshal a bodies cam samples-per-px max-depth opts)
          cap  (+ 64 (* 12 w h))                           ; "255 255 255\n" per pixel + header
          out  (.allocate a cap 16)
          len  (.allocate a 8 8)]
      (check! (.invokeWithArguments rtclj-render-multi-ppm
                                    [scene camera params
                                     (.allocateFrom a ValueLayout/JAVA_INT (int-array devices)) (int (count devices))
                                     out cap len MemorySegment/NULL]))
      (with-open [o (java.io.FileOutputStream. path)]
        (.write (.getChannel o) (.asByteBuffer (.asSlice out 0 (.get len ValueLayout/JAVA_LONG 0))))))))

(defn render-png!
  "render-ppm! with ppm->png (raytracing.clj:176) in place of the P3 text: the render loop on :devices (default
   [0]), then the device PNG writer on the first of them (filtered rows, run-length deflate; DESIGN.md section
   4.11).  The compressed file comes back and is handed to a single .write; its pixels are those of scene.ppm."
  [^String path bodies cam samples-per-px max-depth & {:keys [devices] :or {devices [0]} :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [[scene camera params] (marshal a bodies cam samples-per-px max-depth opts)
          devs (.allocateFrom a ValueLayout/JAVA_INT (int-array devices))
          len  (.allocate a 8 8)
          _    (check! (.invokeWithArguments rtclj-render-multi-png          ; sizing call: nothing is rendered
                                             [scene camera params devs (int (count devices))
                                              MemorySegment/NULL 0 len MemorySegment/NULL]))
          cap  (.get len ValueLayout/JAVA_LONG 0)
          out  (.allocate a cap 16)]
      (check! (.invokeWithArguments rtclj-render-multi-png
                                    [scene camera params devs (int (count devices)) out cap len MemorySegment/NULL]))
      (with-open [o (java.io.FileOutputStream. path)]
        (.write (.getChannel o) (.asByteBuffer (.asSlice out 0 (.get len ValueLayout/JAVA_LONG 0))))))))

(defn render-into-realm!
  "realm.raytracing: copies the linear image into realm[0 .. 3*W*H) where the reference's loop
   (realm/raytracing.clj:325-346) leaves it, so its PPM block (:350-358) can stay."
  [^doubles realm bodies cam samples-per-px max-depth & opts]
  (let [colors (apply render bodies cam samples-per-px max-depth :flags flags-realm opts)]
    (dotimes [p (count colors)]
      (let [^doubles c (nth colors p)]
        (aset realm (* 3 p) (aget c 0))
        (aset realm (+ 1 (* 3 p)) (aget c 1))
        (aset realm (+ 2 (* 3 p)) (aget c 2))))
    realm))

;; ---- progressive rendering: the same loop in passes, an image that refines (rtclj_progressive_*)
;; int rtclj_progressive_create(const rtclj_scene*, const rtclj_camera*, const rtclj_params*,
;;                              const int32_t* devices, int32_t n_devices, int32_t* pass_unit,
;;                              rtclj_progressive** out)
(def ^:private rtclj-progressive-create
  (downcall "rtclj_progressive_create"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS)))
;; int rtclj_progressive_step(rtclj_progressive*, int32_t samples, double* out_linear, uint8_t* out_rgb8,
;;                            int32_t* samples_done, rtclj_stats*)
(def ^:private rtclj-progressive-step
  (downcall "rtclj_progressive_step"
            (fd-int ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/ADDRESS ValueLayout/ADDRESS)))
;; int rtclj_progressive_destroy(rtclj_progressive*)
(def ^:private rtclj-progressive-destroy
  (downcall "rtclj_progressive_destroy" (fd-int ValueLayout/ADDRESS)))

;; ---- adaptive sampling: passes trace only the pixels whose noise is still above a tolerance (DESIGN.md 4.10)
;; int rtclj_progressive_create_adaptive(const rtclj_scene*, const rtclj_camera*, const rtclj_params*,
;;                                       const double tolerance[2], int32_t min_samples, const int32_t* devices,
;;                                       int32_t n_devices, int32_t* pass_unit, rtclj_progressive** out)
(def ^:private rtclj-progressive-create-adaptive
  (downcall "rtclj_progressive_create_adaptive"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS
                    ValueLayout/ADDRESS)))
;; int rtclj_progressive_noise(rtclj_progressive*, int32_t* samples, double* noise, uint64_t* active_pixels)
(def ^:private rtclj-progressive-noise
  (downcall "rtclj_progressive_noise"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS)))

(defn- pinned-bytes
  "n bytes of PINNED host memory (rtclj_host_alloc).  Returns [segment free-fn]."
  [^Arena a ^long n]
  (let [slot (.allocate a 8 8)
        _    (check! (.invokeWithArguments rtclj-host-alloc [n slot]))
        ^MemorySegment p (.reinterpret (.get slot ValueLayout/ADDRESS 0) n)]
    [p #(.invokeWithArguments rtclj-host-free [p])]))

(defn progressive
  "Begins a progressive render: the compute-pixel loop (raytracing.clj:141-171) run in passes towards
   samples-per-px samples, on :devices (default [0]), with the options of `render`.  After passes totalling
   d samples the image is bit-identical to `render` with d samples in the same summation order.  Returns a
   handle map; :pass-unit is the granularity of passes (every pass but the last a multiple of it).  Close it
   with progressive-close!."
  [bodies cam samples-per-px max-depth & {:keys [devices] :or {devices [0]} :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [w    (long (:image-width cam))
          h    (long (:image-height cam))
          [scene camera params] (marshal a bodies cam samples-per-px max-depth opts)
          unit (.allocate a 4 4)
          slot (.allocate a 8 8)]
      (check! (.invokeWithArguments rtclj-progressive-create
                                    [scene camera params
                                     (.allocateFrom a ValueLayout/JAVA_INT (int-array devices)) (int (count devices))
                                     unit slot]))
      (let [handle (.get slot ValueLayout/ADDRESS 0)]
        (try
          (let [[linear free-linear!] (pinned-doubles a (* 3 w h))
                [rgb8 free-rgb8!]     (pinned-bytes a (* 3 w h))]
            {:handle handle :pass-unit (.get unit ValueLayout/JAVA_INT 0) :samples-per-px samples-per-px
             :linear linear :rgb8 rgb8 :free! (fn [] (free-linear!) (free-rgb8!))})
          (catch Throwable t
            (.invokeWithArguments rtclj-progressive-destroy [handle])
            (throw t)))))))

(declare progressive-close!)

(defn progressive-adaptive
  "Begins an adaptive progressive render: `progressive`, but every pass traces only the pixels whose noise
   estimate (the standard error of the pixel mean, per channel) is still above abs-tol + rel-tol * |mean|, after
   at least :min-samples samples (at least two pass units; default exactly two).  A pixel that stops keeps its
   image, bit-identical to `render` with its own sample count.  Use progressive-step!, progressive-noise and
   progressive-close! on the handle."
  [bodies cam samples-per-px max-depth abs-tol rel-tol & {:keys [devices min-samples] :or {devices [0]} :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [w    (long (:image-width cam))
          h    (long (:image-height cam))
          [scene camera params] (marshal a bodies cam samples-per-px max-depth opts)
          tol  (.allocateFrom a ValueLayout/JAVA_DOUBLE (double-array [abs-tol rel-tol]))
          unit (.allocate a 4 4)
          slot (.allocate a 8 8)
          create (fn [least]
                   (.invokeWithArguments rtclj-progressive-create-adaptive
                                         [scene camera params tol (int least)
                                          (.allocateFrom a ValueLayout/JAVA_INT (int-array devices)) (int (count devices))
                                          unit slot]))]
      ;; the default minimum is two pass units: the unit comes from a plain create of the same params
      (if min-samples
        (check! (create min-samples))
        (let [probe (progressive bodies cam samples-per-px max-depth opts)
              least (* 2 (:pass-unit probe))]
          (progressive-close! probe)
          (check! (create least))))
      (let [handle (.get slot ValueLayout/ADDRESS 0)]
        (try
          (let [[linear free-linear!] (pinned-doubles a (* 3 w h))
                [rgb8 free-rgb8!]     (pinned-bytes a (* 3 w h))]
            {:handle handle :pass-unit (.get unit ValueLayout/JAVA_INT 0) :samples-per-px samples-per-px
             :width w :height h :linear linear :rgb8 rgb8 :free! (fn [] (free-linear!) (free-rgb8!))})
          (catch Throwable t
            (.invokeWithArguments rtclj-progressive-destroy [handle])
            (throw t)))))))

;; ---- accumulations over frames: a camera sequence accumulated in shared launches (DESIGN.md 4.15)
;; int rtclj_progressive_create_frames(const rtclj_scene*, const rtclj_camera* cameras, int32_t n_frames,
;;                                     const rtclj_params*, const double* tolerance, int32_t min_samples,
;;                                     const int32_t* devices, int32_t n_devices, int32_t* pass_unit,
;;                                     rtclj_progressive** out)
(def ^:private rtclj-progressive-create-frames
  (downcall "rtclj_progressive_create_frames"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS
                    ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT
                    ValueLayout/ADDRESS ValueLayout/ADDRESS)))

(defn- progressive-frames*
  "rtclj_progressive_create_frames with tolerance `tol` ([abs rel], or nil: plain) and min-samples `least`."
  [bodies cams samples-per-px max-depth tol least {:keys [devices] :or {devices [0]} :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [cam0    (first cams)
          w       (long (:image-width cam0))
          h       (long (:image-height cam0))
          k       (count cams)
          [scene _ params] (marshal a bodies cam0 samples-per-px max-depth opts)
          cameras (.allocate a (* (max k 1) (size :rtclj_camera)) 8)
          _       (doseq [[i cam] (map-indexed vector cams)]
                    (fill-camera! (.asSlice cameras (* i (size :rtclj_camera)) (size :rtclj_camera)) cam))
          unit    (.allocate a 4 4)
          slot    (.allocate a 8 8)]
      (check! (.invokeWithArguments rtclj-progressive-create-frames
                                    [scene cameras (int k) params
                                     (if tol (.allocateFrom a ValueLayout/JAVA_DOUBLE (double-array tol)) MemorySegment/NULL)
                                     (int least)
                                     (.allocateFrom a ValueLayout/JAVA_INT (int-array devices)) (int (count devices))
                                     unit slot]))
      (let [handle (.get slot ValueLayout/ADDRESS 0)]
        (try
          (let [[linear free-linear!] (pinned-doubles a (* 3 w h k))
                [rgb8 free-rgb8!]     (pinned-bytes a (* 3 w h k))]
            {:handle handle :pass-unit (.get unit ValueLayout/JAVA_INT 0) :samples-per-px samples-per-px
             :width w :height h :frames k :linear linear :rgb8 rgb8 :free! (fn [] (free-linear!) (free-rgb8!))})
          (catch Throwable t
            (.invokeWithArguments rtclj-progressive-destroy [handle])
            (throw t)))))))

(defn progressive-frames
  "Begins a progressive render of a camera sequence (`cams`, camera maps of one image size, as render-frames takes
   them): all frames accumulate in shared launches, and after every step frame f is bit-identical to (progressive
   bodies (nth cams f) ...) stepped alike.  Use progressive-step! (its images hold the frames one after the other,
   W*H*3 values each) and progressive-close! on the handle."
  [bodies cams samples-per-px max-depth & {:as opts}]
  (progressive-frames* bodies cams samples-per-px max-depth nil 0 opts))

(defn progressive-frames-adaptive
  "progressive-frames with adaptive sampling: every pass traces only the pixels of every frame whose noise estimate
   is still above abs-tol + rel-tol * |mean| (see progressive-adaptive, whose :min-samples default it shares); frame f
   is bit-identical to (progressive-adaptive bodies (nth cams f) ...) stepped alike.  progressive-noise returns the
   frames' sample counts and noise one after the other and the active pixels of all frames."
  [bodies cams samples-per-px max-depth abs-tol rel-tol & {:keys [min-samples] :as opts}]
  (let [least (or min-samples
                  (let [probe (progressive-frames bodies (take 1 cams) samples-per-px max-depth opts)]
                    (try (* 2 (:pass-unit probe)) (finally (progressive-close! probe)))))]
    (progressive-frames* bodies cams samples-per-px max-depth [abs-tol rel-tol] least opts)))

(defn progressive-noise
  "After a step of a progressive-adaptive render: {:samples int[W*H], the samples each pixel has, :stderr
   double[W*H*3], its noise estimate, :active, the pixels the next pass traces (0: the render is done)}.  A render of
   frames returns every frame's, one after the other."
  [p]
  (with-open [a (Arena/ofConfined)]
    (let [n       (* (long (:width p)) (long (:height p)) (long (:frames p 1)))
          samples (.allocate a (* 4 n) 8)
          stderr  (.allocate a (* 24 n) 8)
          active  (.allocate a 8 8)]
      (check! (.invokeWithArguments rtclj-progressive-noise [(:handle p) samples stderr active]))
      {:samples (.toArray samples ValueLayout/JAVA_INT)
       :stderr  (.toArray stderr ValueLayout/JAVA_DOUBLE)
       :active  (.get active ValueLayout/JAVA_LONG 0)})))

(defn progressive-step!
  "One pass of `samples` samples per pixel.  Returns {:linear :rgb8 :samples-done}: the image so far as
   W*H*3 doubles (linear RGB, row-major from the top-left pixel) and W*H*3 bytes quantised like write-color!,
   both in PINNED memory that belongs to `p`: the next step overwrites them, progressive-close! frees them."
  [p samples]
  (with-open [a (Arena/ofConfined)]
    (let [done (.allocate a 4 4)]
      (check! (.invokeWithArguments rtclj-progressive-step
                                    [(:handle p) (int samples) (:linear p) (:rgb8 p) done MemorySegment/NULL]))
      {:linear (:linear p) :rgb8 (:rgb8 p) :samples-done (.get done ValueLayout/JAVA_INT 0)})))

(defn progressive-close!
  "Ends a progressive render: its GPU contexts and its pinned images are released."
  [p]
  (try
    (check! (.invokeWithArguments rtclj-progressive-destroy [(:handle p)]))
    (finally ((:free! p)))))

;; int rtclj_encode_ppm_p3_gpu(int32_t device, const uint8_t* rgb8, int32_t width, int32_t height,
;;                             char* out, size_t capacity, size_t* len)
(def ^:private rtclj-encode-ppm-p3-gpu
  (downcall "rtclj_encode_ppm_p3_gpu"
            (fd-int ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/JAVA_INT
                    ValueLayout/ADDRESS ValueLayout/JAVA_LONG ValueLayout/ADDRESS)))

(defn write-ppm!
  "The write-color! loop (raytracing.clj:172-175) as ONE call: rgb8 is a byte[] of W*H*3 gamma-encoded
   components (what write-color! computes per pixel; rtclj_render fills it when asked for out_rgb8);
   the P3 text is produced by the device kernels and handed to a single .write."
  [^String path ^bytes rgb8 width height & {:keys [device] :or {device 0}}]
  (with-open [a (Arena/ofConfined)]
    (let [w     (int width) h (int height)
          src   (.allocateFrom a ValueLayout/JAVA_BYTE rgb8)
          cap   (+ 64 (* 12 (long w) (long h)))            ; "255 255 255\n" per pixel + header
          out   (.allocate a cap 16)
          len   (.allocate a 8 8)]
      (check! (.invokeWithArguments rtclj-encode-ppm-p3-gpu [(int device) src w h out cap len]))
      (let [n (.get len ValueLayout/JAVA_LONG 0)]
        (with-open [o (java.io.FileOutputStream. path)]
          (.write (.getChannel o) (.asByteBuffer (.asSlice out 0 n))))))))

;; int rtclj_encode_png_gpu(int32_t device, const uint8_t* rgb8, int32_t width, int32_t height,
;;                          uint8_t* out, size_t capacity, size_t* len)
(def ^:private rtclj-encode-png-gpu
  (downcall "rtclj_encode_png_gpu"
            (fd-int ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/JAVA_INT
                    ValueLayout/ADDRESS ValueLayout/JAVA_LONG ValueLayout/ADDRESS)))

(defn encode-png-gpu
  "ppm->png's writer (raytracing.clj:176) on the GPU: rgb8 is a byte[] of W*H*3 components (row-major from the
   top-left pixel), the result a byte[] holding a compressed PNG of it (DESIGN.md section 4.11)."
  ^bytes [^bytes rgb8 width height & {:keys [device] :or {device 0}}]
  (with-open [a (Arena/ofConfined)]
    (let [w   (int width) h (int height)
          src (.allocateFrom a ValueLayout/JAVA_BYTE rgb8)
          len (.allocate a 8 8)
          _   (check! (.invokeWithArguments rtclj-encode-png-gpu [(int device) src w h MemorySegment/NULL 0 len]))
          cap (.get len ValueLayout/JAVA_LONG 0)
          out (.allocate a cap 16)]
      (check! (.invokeWithArguments rtclj-encode-png-gpu [(int device) src w h out cap len]))
      (.toArray (.asSlice out 0 (.get len ValueLayout/JAVA_LONG 0)) ValueLayout/JAVA_BYTE))))

;; ---- animated PNG of a camera sequence (DESIGN.md section 4.14)
;; int rtclj_encode_apng_gpu(int32_t device, const uint8_t* frames, int32_t width, int32_t height, int32_t n_frames,
;;                           int32_t delay_num, int32_t delay_den, int32_t plays, uint8_t* out, size_t capacity,
;;                           size_t* len)
(def ^:private rtclj-encode-apng-gpu
  (downcall "rtclj_encode_apng_gpu"
            (fd-int ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/JAVA_INT ValueLayout/JAVA_INT
                    ValueLayout/JAVA_INT ValueLayout/JAVA_INT ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_LONG
                    ValueLayout/ADDRESS)))
;; int rtclj_render_frames_apng(const rtclj_scene*, const rtclj_camera* cameras, int32_t n_frames, const rtclj_params*,
;;                              int32_t delay_num, int32_t delay_den, int32_t plays, const int32_t* devices,
;;                              int32_t n_devices, uint8_t* out, size_t capacity, size_t* len, rtclj_stats*)
(def ^:private rtclj-render-frames-apng
  (downcall "rtclj_render_frames_apng"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT
                    ValueLayout/JAVA_INT ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS
                    ValueLayout/JAVA_LONG ValueLayout/ADDRESS ValueLayout/ADDRESS)))

(defn encode-apng-gpu
  "An animated PNG of n-frames frames on the GPU: rgb8 is a byte[] of n-frames consecutive W*H*3 images (row-major
   from the top-left pixel), the result a byte[] whose every frame carries the compressed PNG data encode-png-gpu
   writes for it.  :delay [num den] seconds per frame (default [1 30]), :plays loops (default 0: forever)."
  ^bytes [^bytes rgb8 width height n-frames & {:keys [device delay plays] :or {device 0 delay [1 30] plays 0}}]
  (with-open [a (Arena/ofConfined)]
    (let [[num den] delay
          args (fn [out cap len] [(int device) (.allocateFrom a ValueLayout/JAVA_BYTE rgb8) (int width) (int height)
                                  (int n-frames) (int num) (int den) (int plays) out (long cap) len])
          len  (.allocate a 8 8)
          _    (check! (.invokeWithArguments rtclj-encode-apng-gpu (args MemorySegment/NULL 0 len)))
          cap  (.get len ValueLayout/JAVA_LONG 0)
          out  (.allocate a cap 16)]
      (check! (.invokeWithArguments rtclj-encode-apng-gpu (args out cap len)))
      (.toArray (.asSlice out 0 (.get len ValueLayout/JAVA_LONG 0)) ValueLayout/JAVA_BYTE))))

(defn render-frames-apng!
  "render-frames and encode-apng-gpu as ONE native call (rtclj_render_frames_apng): the camera sequence `cams` rendered
   on :devices (default [0]), every frame assembled on the first of them and encoded there as one animated PNG, which
   comes back and is handed to a single .write.  Options as render-frames, plus :delay [num den] (default [1 30]) and
   :plays (default 0: loop forever)."
  [^String path bodies cams samples-per-px max-depth
   & {:keys [devices delay plays] :or {devices [0] delay [1 30] plays 0} :as opts}]
  (with-open [a (Arena/ofConfined)]
    (let [k       (count cams)
          [scene _ params] (marshal a bodies (first cams) samples-per-px max-depth opts)
          cameras (.allocate a (* k (size :rtclj_camera)) 8)
          _       (doseq [[i cam] (map-indexed vector cams)]
                    (fill-camera! (.asSlice cameras (* i (size :rtclj_camera)) (size :rtclj_camera)) cam))
          devs    (.allocateFrom a ValueLayout/JAVA_INT (int-array devices))
          [num den] delay
          args    (fn [out cap len] [scene cameras (int k) params (int num) (int den) (int plays) devs
                                     (int (count devices)) out (long cap) len MemorySegment/NULL])
          len     (.allocate a 8 8)
          _       (check! (.invokeWithArguments rtclj-render-frames-apng (args MemorySegment/NULL 0 len)))  ; sizing
          cap     (.get len ValueLayout/JAVA_LONG 0)
          out     (.allocate a cap 16)]
      (check! (.invokeWithArguments rtclj-render-frames-apng (args out cap len)))
      (with-open [o (java.io.FileOutputStream. path)]
        (.write (.getChannel o) (.asByteBuffer (.asSlice out 0 (.get len ValueLayout/JAVA_LONG 0))))))))

;; ---- denoising (DESIGN.md section 4.13): an edge-avoiding filter guided by the normal-shaded primary render
;; int rtclj_denoise_gpu(int32_t device, const double* linear, const double* guide, int32_t width, int32_t height,
;;                       int32_t levels, const double sigma[2], uint32_t flags, double* out_linear, uint8_t* out_rgb8)
(def ^:private rtclj-denoise-gpu
  (downcall "rtclj_denoise_gpu"
            (fd-int ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/JAVA_INT
                    ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS)))
;; int rtclj_render_denoised(const rtclj_scene*, const rtclj_camera*, const rtclj_params*, int32_t guide_samples,
;;                           int32_t levels, const double sigma[2], const int32_t* devices, int32_t n_devices,
;;                           double* out_linear, uint8_t* out_rgb8, rtclj_stats*)
(def ^:private rtclj-render-denoised
  (downcall "rtclj_render_denoised"
            (fd-int ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/JAVA_INT
                    ValueLayout/ADDRESS ValueLayout/ADDRESS ValueLayout/JAVA_INT ValueLayout/ADDRESS ValueLayout/ADDRESS
                    ValueLayout/ADDRESS)))

(def denoise-defaults
  "levels, sigma-color, sigma-guide and guide samples chosen by the sweep of DESIGN.md section 4.13 (the Python
   defaults, render.DENOISE_*)."
  {:levels 3 :sigma-color 0.5 :sigma-guide 0.4 :guide-samples 4})

(defn- colors-of
  "W*H double[3] pixels of a W*H*3 double segment, as `render` returns them."
  [^MemorySegment out ^long n]
  (mapv (fn [^long p]
          (double-array [(.getAtIndex out ValueLayout/JAVA_DOUBLE (* 3 p))
                         (.getAtIndex out ValueLayout/JAVA_DOUBLE (+ 1 (* 3 p)))
                         (.getAtIndex out ValueLayout/JAVA_DOUBLE (+ 2 (* 3 p)))]))
        (range n)))

(defn denoise
  "The filter alone on GPU :device (default 0): `colors` and `guide` are what `render` returns (W*H double[3], the
   guide rendered with :flags flags-i, max-depth 1 and the same seed).  Returns the denoised pixels in the same form."
  [colors guide width height & {:keys [device levels sigma-color sigma-guide flags]
                                :or {device 0 flags 0} :as opts}]
  (let [{:keys [levels sigma-color sigma-guide]} (merge denoise-defaults (select-keys opts [:levels :sigma-color :sigma-guide]))]
    (with-open [a (Arena/ofConfined)]
      (let [n   (* (long width) (long height))
            lin (doubles-seg a (mapcat seq colors))
            gd  (doubles-seg a (mapcat seq guide))
            out (.allocate a (* 24 n) 8)]
        (check! (.invokeWithArguments rtclj-denoise-gpu
                                      [(int device) lin gd (int width) (int height) (int levels)
                                       (doubles-seg a [sigma-color sigma-guide]) (int flags) out MemorySegment/NULL]))
        (colors-of out n)))))

(defn render-denoised
  "`render` followed by the denoiser, in one native call (rtclj_render_denoised): the colour render on :devices
   (default [0]), the guide (the same camera and seed, :guide-samples samples, max-depth 1, normal shading), both
   assembled on the first device and filtered there.  Options as `render`, plus :guide-samples :levels :sigma-color
   :sigma-guide (defaults: denoise-defaults).  Returns the denoised pixels as `render` returns its image."
  [bodies cam samples-per-px max-depth & {:keys [devices] :or {devices [0]} :as opts}]
  (let [{:keys [guide-samples levels sigma-color sigma-guide]} (merge denoise-defaults opts)]
    (with-open [a (Arena/ofConfined)]
      (let [n (* (long (:image-width cam)) (long (:image-height cam)))
            [scene camera params] (marshal a bodies cam samples-per-px max-depth opts)
            [^MemorySegment out free!] (pinned-doubles a (* 3 n))]
        (try
          (check! (.invokeWithArguments rtclj-render-denoised
                                        [scene camera params (int guide-samples) (int levels)
                                         (doubles-seg a [sigma-color sigma-guide])
                                         (.allocateFrom a ValueLayout/JAVA_INT (int-array devices)) (int (count devices))
                                         out MemorySegment/NULL MemorySegment/NULL]))
          (colors-of out n)
          (finally (free!)))))))
