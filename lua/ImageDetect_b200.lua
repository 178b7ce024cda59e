--[[ ImageDetect_b200.lua — fbcoco.ImageDetect (ImageDetect.lua:9-193) whose forward runs in libmpn_b200.so.

The contract is the reference's, argument for argument, so that Tester_FRCNN.lua:24,38-49,72,86 and demo.lua:43,75 need
NO edit:
   fbcoco.ImageDetect(model, transformer, scale, max_size)   model = the nn.Sequential a model file returns / torch.load
   :detect(im, boxes, min_images, recompute_features)        -> FloatTensor R x C, FloatTensor R x 4C   (:156-193)
   :computeRawOutputs(im, boxes, min_images, recompute_features) -> {class, bbox} as model:forward returns (:137-153)
   :memoryEfficientForward(model, input, bs, recompute_features) -> {CudaTensor R x C, CudaTensor R x 4C} (:91-135)
`self.model` stays the nn module (Tester_FRCNN.lua:37-49 calls module:apply, a dummy module:forward and reads
module.output[1]:size(2) on it; train.lua keeps training it). The mpn_model built from its graph (lua/model_desc.lua,
weights copied once) lives in a weak-keyed table OUTSIDE every serialisable field — torch.save / clearState never see a
C handle — and is dropped when the module is cleared (nn.Module.clearState hook below) or was put back into training
mode since the last detect (its weights may have moved: train.lua tests the module it trains).

getImages runs in Lua exactly as in the reference by default; with `mpn_getimages=device` in the environment the raw
image goes to mpn_model_trunk_image, which applies the transformer and image.scale on the GPU (SURVEY 8f-1).
UNTESTED in the build environment (no Torch-7 there): tests/test_lua_shim_cpu.py checks the class surface, the
constructor arity and every C call against include/mpn_abi.h. ]]
local ffi = require 'ffi'
local mpn = paths.dofile('mpn_ffi.lua')
local model_desc = paths.dofile('model_desc.lua')
local C = mpn.C
local ImageDetect = torch.class('fbcoco.ImageDetect')

-- nn module -> {handle = mpn_model* (ffi.gc'd), num_classes}; weak keys: a collected module frees its mpn_model
local handles = setmetatable({}, {__mode = 'k'})
if not nn.Module._mpn_clear_hooked then
   local clearState = nn.Module.clearState
   function nn.Module:clearState()
      handles[self] = nil                                   -- model:clearState() before torch.save (train.lua:193-195)
      return clearState(self)
   end
   nn.Module._mpn_clear_hooked = true
end

function ImageDetect:__init(model, transformer, scale, max_size)
   assert(model, 'must provide model!')
   assert(transformer, 'must provide transformer!')
   self.model = model
   self.image_transformer = transformer
   self.scale = scale or {600}
   self.max_size = max_size or 1000
end

-- the mpn_model of self.model, (re)built lazily
local function native(self)
   local m = self.model
   if m.train ~= false then handles[m] = nil end            -- in training mode since the last detect: weights may differ
   local h = handles[m]
   if not h then
      h = model_desc.create(m, {max_rois = tonumber(os.getenv('mpn_max_rois')) or 4096,
                                max_h = tonumber(os.getenv('mpn_max_h')) or 1024, max_w = tonumber(os.getenv('mpn_max_w')) or 1344})
      handles[m] = h
   end
   m:evaluate()                                             -- ImageDetect.lua:157 (also marks the handle as current)
   return h
end
ImageDetect._native = native                                -- lua/Tester_b200.lua uses the same handle

local function getImage(self, im)   -- ImageDetect.lua:22-52, single scale
   im = self.image_transformer:forward(im)
   local s = im[1]:size()
   local smin, smax = math.min(s[1], s[2]), math.max(s[1], s[2])
   local im_scale = self.scale[1] / smin
   if torch.round(im_scale * smax) > self.max_size then im_scale = self.max_size / smax end
   return image.scale(im, s[2] * im_scale, s[1] * im_scale):float():contiguous(), im_scale
end
ImageDetect._getImage = getImage

local function project_im_rois(boxes, im_scale)            -- ImageDetect.lua:54-73, single scale
   local rois = torch.FloatTensor(boxes:size(1), 5)
   rois[{{}, 1}]:fill(1)
   rois[{{}, {2, 5}}]:copy(boxes):add(-1):mul(im_scale):add(1)
   return rois
end

local on_device = os.getenv('mpn_getimages') == 'device'
local function transform_struct(t)   -- fbcoco.ImageTransformer fields (ImageTransformer.lua:11-17) -> mpn_image_transform
   local tf = ffi.new('mpn_image_transform')
   for i = 1, 3 do
      tf.swap[i - 1] = t.swap and t.swap[i] or i
      tf.mean[i - 1] = t.mean[i]
      tf.std[i - 1] = t.std and t.std[i] or 1
   end
   tf.scale = t.scale or 1
   tf.has_std = t.std and 1 or 0
   return tf
end
ImageDetect._transform_struct = transform_struct

-- ImageDetect.lua:91-135. input = {images N x 3 x H x W, rois R x 5}, CudaTensors (what detect / the Tester hand over).
-- The trunk runs once, the heads on ALL rois in one pass: the reference chunks by `bs` only to bound memory, and its own
-- self-test (:126-133) demands chunked == unchunked exactly, which the library guarantees (row-chunk invariance), so
-- `bs` is accepted and ignored. Device pointers go straight through: no host round trip.
function ImageDetect:memoryEfficientForward(model, input, bs, recompute_features)
   local images, rois = input[1], input[2]
   if recompute_features == nil then recompute_features = true end
   assert(model == self.model, 'memoryEfficientForward: model must be the detector\'s own module')
   local h = native(self)
   local R, nc = rois:size(1), h.num_classes
   assert(images:isContiguous() and rois:isContiguous() and rois:size(2) == 5)
   assert(torch.type(images) == 'torch.CudaTensor' and torch.type(rois) == 'torch.CudaTensor', 'expects CudaTensors (ImageDetect.lua:146-150)')
   -- assuming the net has bbox regression part (ImageDetect.lua:101)
   self.output = self.output or {torch.CudaTensor(), torch.CudaTensor()}
   self.output[1]:resize(R, nc)
   self.output[2]:resize(R, nc * 4)
   local ctx = mpn.ctx()
   if recompute_features then
      assert(images:size(1) >= 1 and images:size(2) == 3)
      if images:size(1) == 1 then
         mpn.check(ctx, C.mpn_model_trunk_dev(h.handle, mpn.fptr(images), images:size(3), images:size(4)), 'mpn_model_trunk_dev')
      else   -- a padded batch: every image goes through the trunk, ROI rows pick theirs with column 1 (1-based)
         mpn.check(ctx, C.mpn_model_trunk_batch_dev(h.handle, mpn.fptr(images), images:size(1), images:size(3), images:size(4)),
                   'mpn_model_trunk_batch_dev')
      end
   end
   mpn.check(ctx, C.mpn_model_heads_dev(h.handle, mpn.fptr(rois), R, mpn.fptr(self.output[1]), mpn.fptr(self.output[2])), 'mpn_model_heads_dev')
   return self.output
end

-- ImageDetect.lua:137-153: the network's own outputs for one image (class R x C: logits, or probabilities for an integral
-- head; bbox R x 4C after BBoxNorm), as CudaTensors like model:forward
function ImageDetect:computeRawOutputs(im, boxes, min_images, recompute_features)
   local h = native(self)
   local img, im_scale = getImage(self, im)
   self._im_scale = im_scale
   local rois = project_im_rois(boxes:float(), im_scale)
   self.inputs_cuda = self.inputs_cuda or {torch.CudaTensor(), torch.CudaTensor()}
   self.inputs_cuda[1]:resize(1, 3, img:size(2), img:size(3)):copy(img)
   self.inputs_cuda[2]:resize(rois:size()):copy(rois)
   return self:memoryEfficientForward(self.model, self.inputs_cuda, 500, true)
end

-- supposes boxes is in [x1,y1,x2,y2] format
function ImageDetect:detect(im, boxes, min_images, recompute_features)
   if recompute_features == nil then recompute_features = true end
   local h = native(self)
   local b = boxes:float():contiguous()
   local R, nc = b:size(1), h.num_classes
   local img, im_scale
   if recompute_features and on_device then
      local raw = im:float():contiguous()
      local s, hh, ww = ffi.new('double[1]'), ffi.new('int32_t[1]'), ffi.new('int32_t[1]')
      mpn.check(mpn.ctx(), C.mpn_model_trunk_image(h.handle, mpn.fptr(raw), raw:size(2), raw:size(3),
                transform_struct(self.image_transformer), self.scale[1], self.max_size, s, hh, ww), 'mpn_model_trunk_image')
      im_scale = s[0]; self._im_scale = im_scale
      recompute_features = false                      -- the trunk has run: heads on the cached features
   elseif recompute_features then
      img, im_scale = getImage(self, im); self._im_scale = im_scale
   else
      im_scale = self._im_scale
   end
   local scores, bboxes = torch.FloatTensor(R, nc), torch.FloatTensor(R, 4 * nc)
   local rc = C.mpn_model_detect(h.handle, img and mpn.fptr(img) or nil, img and img:size(2) or 0, img and img:size(3) or 0,
                                 mpn.fptr(b), R, im_scale, recompute_features and 1 or 0, mpn.fptr(scores), mpn.fptr(bboxes))
   mpn.check(mpn.ctx(), rc, 'mpn_model_detect')
   return scores, bboxes
end
